// tcgen05.cuh — PTX wrappers of the 5th-gen tensor-core engines (tcgen05 / TMEM / mbarriers, sm_100a) and the streamed
// weight-slot format, shared by epic_tc.cu, epic_wide_tc.cu and absorb_head_tc.cu.
#pragma once

#include <cuda_bf16.h>
#include <stddef.h>
#include <stdint.h>

#include <vector>

namespace mmb {

// ---- PTX wrappers ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// 1-D TMA: global -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (bf16 in, fp32 accumulate); one thread issues
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// shared-memory matrix descriptor, no swizzle (SURVEY/DESIGN: bits 0-13 addr>>4, 16-29 LBO>>4,
// 32-45 SBO>>4, 46-47 version=1, 61-63 layout=0)
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | ((uint64_t)1 << 46);
}
// instruction descriptor kind::f16: D fp32 (bit 4), A/B bf16 (bits 7,10), N>>3 at 17, M>>4 at 24; b_mn = B is MN-major
__host__ __device__ constexpr uint32_t instr_desc(int M, int N, bool b_mn = false) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (b_mn ? (1u << 16) : 0u) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}

// [128 rows x 128 k] bf16 tile, K-major canonical: 8-row groups 2048 B apart (SBO), 16-byte k-chunks 128 B apart (LBO).
// thread `row` stores columns [col, col + CW) of its row
template <int CW>
__device__ __forceinline__ void store_row(uint8_t* tile, int row, int col, const float (&v)[CW]) {
    uint8_t* p = tile + (row >> 3) * 2048 + (row & 7) * 16 + (col >> 3) * 128;
#pragma unroll
    for (int c = 0; c < CW / 8; ++c)
        *reinterpret_cast<uint4*>(p + c * 128) = make_uint4(pack_bf16(v[8 * c], v[8 * c + 1]), pack_bf16(v[8 * c + 2], v[8 * c + 3]),
                                                            pack_bf16(v[8 * c + 4], v[8 * c + 5]), pack_bf16(v[8 * c + 6], v[8 * c + 7]));
}

// Sum `vals[0..CNT)` over the 32 lanes of a warp by recursive halving: each stage exchanges half of the values a lane still
// holds (CNT-1 shuffles in total instead of 5*CNT).  On return lane l holds, in vals[0], the warp total of the value whose index
// has bit log2(CNT/2) = lane bit 4, ..., i.e. idx = sum_k ((l >> (4-k)) & 1) * (CNT >> (k+1)); CNT <= 32, a power of two.
template <int CNT>
__device__ __forceinline__ void warp_halving_sum(float (&vals)[CNT], int lane) {
    int off = 16;
#pragma unroll
    for (int cnt = CNT; cnt > 1; cnt >>= 1, off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < cnt / 2; ++i) {
            const float keep = upper ? vals[cnt / 2 + i] : vals[i];
            const float send = upper ? vals[i] : vals[cnt / 2 + i];
            vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    for (; off >= 1; off >>= 1) vals[0] += __shfl_xor_sync(0xffffffffu, vals[0], off);
}
template <int CNT>
__device__ __forceinline__ int warp_halving_index(int lane) {
    int idx = 0, off = 16;
#pragma unroll
    for (int cnt = CNT; cnt > 1; cnt >>= 1, off >>= 1) idx += (lane & off) ? cnt / 2 : 0;
    return idx;
}

// ---- streamed weight slot ----------------------------------------------------------------------------------------------------
// One Linear [128 out x 128 k] as the engines stream it L2 -> shared memory (1-D TMA into a two-slot ring, one slot per matrix):
// the bf16 weight tile in the K-major canonical layout (8-row groups 2048 B apart), then at kSlotBias a 4 KB bias tile holding
// each row's bias as hi + lo bf16 in k = 0 and 1 (8-row groups 256 B apart), consumed as one more K-step against a ones tile.
// Where each kernel places the two tiles in shared memory is its own business.
constexpr int kSlot = 36864;        // bytes per slot
constexpr int kSlotBias = 32768;    // byte offset of the bias tile (= bytes of the weight tile)

// element (row o, k) of a K-major tile with 8-row groups `sbo` bytes apart -> bf16 index
inline size_t tile_index(int o, int k, int sbo) { return ((size_t)(o / 8) * sbo + (size_t)(k / 8) * 128 + (o % 8) * 16 + (k % 8) * 2) / 2; }

// host: weight (o, k) of slot s of an image of bf16 slots
inline void slot_put_weight(std::vector<__nv_bfloat16>& img, int s, int o, int k, float w) {
    img[(size_t)s * kSlot / 2 + tile_index(o, k, 2048)] = __float2bfloat16(w);
}
// host: bias of row o of slot s, split into bf16 hi + lo
inline void slot_put_bias(std::vector<__nv_bfloat16>& img, int s, int o, float b) {
    const __nv_bfloat16 hi = __float2bfloat16(b);
    img[(size_t)s * kSlot / 2 + kSlotBias / 2 + tile_index(o, 0, 256)] = hi;
    img[(size_t)s * kSlot / 2 + kSlotBias / 2 + tile_index(o, 1, 256)] = __float2bfloat16(b - __bfloat162float(hi));
}

}  // namespace mmb
