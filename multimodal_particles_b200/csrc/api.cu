// api.cu — the extern "C" surface of libmmbridge.so (include/mmbridge.h): argument checking, error
// text, model lifetime and dispatch to the kernels.  No exceptions cross this boundary.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <new>

#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {

static thread_local char g_error[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
    return code;
}

int cuda_ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return MMB_OK;
    return fail(MMB_ECUDA, "%s: %s", what, cudaGetErrorString(e));
}

// device image of the step table: [n_steps][4] = (bc, cc, sp, 0) then [n_steps][T] temb
static size_t table_floats(int n_steps, int T) { return (size_t)n_steps * (4 + (size_t)T); }

// ---- table cache -------------------------------------------------------------------------------------------------------
// A generation call gets its per-step scalars as HOST arrays (MmbStepTable).  They are a function of the bridge config only,
// so the device image is built once per distinct table and kept on the model handle.  Steady state: hash the host arrays
// (a few KB), find the slot, launch — no allocation, no copy, nothing that blocks the host.  First use of a table: fill the
// slot's page-locked staging buffer and enqueue ONE cudaMemcpyAsync on the caller's stream (buffers grow on demand).  A fifth
// distinct table evicts the oldest slot after a device synchronisation (kernels of any stream may still be reading it).
constexpr int kTableSlots = 4;
struct TableSlot {
    uint64_t hash = 0;
    size_t floats = 0, cap = 0;
    float* dev = nullptr;
    float* pinned = nullptr;
    bool valid = false;
};
struct TableCache {
    std::mutex mu;
    TableSlot slot[kTableSlots];
    int next = 0;
};

// ---- host-buffer pipeline (mmb_generate_host): internal streams and events, created on first use --------------------------
constexpr int kHostStreams = 4, kHostMaxChunks = 16;
struct HostPipe {
    std::mutex mu;
    bool ready = false;
    cudaStream_t stream[kHostStreams] = {};
    cudaEvent_t fork = nullptr, done[kHostMaxChunks] = {};
};

static int host_pipe_init(HostPipe* hp) {
    std::lock_guard<std::mutex> lock(hp->mu);
    if (hp->ready) return MMB_OK;
    for (auto& s : hp->stream)
        if (int rc = cuda_ok(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking), "host pipeline stream")) return rc;
    if (int rc = cuda_ok(cudaEventCreateWithFlags(&hp->fork, cudaEventDisableTiming), "host pipeline event")) return rc;
    for (auto& e : hp->done)
        if (int rc = cuda_ok(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "host pipeline event")) return rc;
    hp->ready = true;
    return MMB_OK;
}

HostPipe* host_pipe_create() { return new (std::nothrow) HostPipe(); }

void host_pipe_destroy(HostPipe* hp) {
    if (!hp) return;
    for (auto s : hp->stream)
        if (s) cudaStreamDestroy(s);
    if (hp->fork) cudaEventDestroy(hp->fork);
    for (auto e : hp->done)
        if (e) cudaEventDestroy(e);
    delete hp;
}

// reference layout <-> device layout: int64 [P] tokens / masks (mbm.py:13-20) <-> uint8; out-of-range tokens raise a flag
// (the reference asserts 0 <= k < S before every jump, bridges.py:111-115)
__global__ void __launch_bounds__(256) narrow_state_kernel(const long long* __restrict__ k64, const long long* __restrict__ m64,
                                                           uint8_t* __restrict__ k8, uint8_t* __restrict__ m8, size_t P, int S,
                                                           int* __restrict__ bad) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (i >= P) return;
    bool oob = false;
    if (i + 1 < P) {
        const longlong2 kk = *reinterpret_cast<const longlong2*>(k64 + i), mm = *reinterpret_cast<const longlong2*>(m64 + i);
        oob = kk.x < 0 || kk.x >= S || kk.y < 0 || kk.y >= S;
        *reinterpret_cast<uchar2*>(k8 + i) = make_uchar2((unsigned char)kk.x, (unsigned char)kk.y);
        *reinterpret_cast<uchar2*>(m8 + i) = make_uchar2(mm.x != 0, mm.y != 0);
    } else {
        const long long kk = k64[i];
        oob = kk < 0 || kk >= S;
        k8[i] = (uint8_t)kk;
        m8[i] = m64[i] != 0;
    }
    if (oob) atomicOr(bad, 1);
}
// direct mode: masks only (the generation kernel reads features and tokens from the host itself), and the reference's
// token-range assertion over ALL tokens, live or not
__global__ void __launch_bounds__(256) narrow_mask_kernel(const long long* __restrict__ m64, uint8_t* __restrict__ m8, size_t P) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (i >= P) return;
    if (i + 1 < P) {
        const longlong2 mm = *reinterpret_cast<const longlong2*>(m64 + i);
        *reinterpret_cast<uchar2*>(m8 + i) = make_uchar2(mm.x != 0, mm.y != 0);
    } else {
        m8[i] = m64[i] != 0;
    }
}
__global__ void __launch_bounds__(256) check_tokens_kernel(const long long* __restrict__ k64, size_t P, int S, int* __restrict__ bad) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (i >= P) return;
    bool oob;
    if (i + 1 < P) {
        const longlong2 kk = *reinterpret_cast<const longlong2*>(k64 + i);
        oob = kk.x < 0 || kk.x >= S || kk.y < 0 || kk.y >= S;
    } else {
        oob = k64[i] < 0 || k64[i] >= S;
    }
    if (oob) atomicOr(bad, 1);
}
__global__ void __launch_bounds__(256) widen_tokens_kernel(const uint8_t* __restrict__ k8, long long* __restrict__ k64, size_t P) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (i >= P) return;
    if (i + 1 < P) {
        const uchar2 kk = *reinterpret_cast<const uchar2*>(k8 + i);
        *reinterpret_cast<longlong2*>(k64 + i) = make_longlong2(kk.x, kk.y);
    } else {
        k64[i] = k8[i];
    }
}

TableCache* table_cache_create() { return new (std::nothrow) TableCache(); }

void table_cache_destroy(TableCache* c) {
    if (!c) return;
    for (TableSlot& s : c->slot) {
        if (s.dev) cudaFree(s.dev);
        if (s.pinned) cudaFreeHost(s.pinned);
    }
    delete c;
}

static uint64_t hash_words(uint64_t h, const void* data, size_t bytes) {
    const unsigned char* p = static_cast<const unsigned char*>(data);
    size_t i = 0;
    for (; i + 8 <= bytes; i += 8) {
        uint64_t w;
        memcpy(&w, p + i, 8);
        h = (h ^ w) * 0x100000001B3ull;
        h ^= h >> 29;
    }
    for (; i < bytes; ++i) h = (h ^ p[i]) * 0x100000001B3ull;
    return h;
}

// Device image with `floats` floats and content hash `hash`; `fill(dst)` writes it into host memory on a miss.
template <typename Fill>
static int table_cache_get(TableCache* c, uint64_t hash, size_t floats, cudaStream_t stream, Fill fill, const float** out) {
    if (!c) return fail(MMB_EINVAL, "model has no table cache");
    std::lock_guard<std::mutex> lock(c->mu);
    for (TableSlot& s : c->slot)
        if (s.valid && s.hash == hash && s.floats == floats) {
            *out = s.dev;
            return MMB_OK;
        }
    TableSlot* s = nullptr;
    for (TableSlot& t : c->slot)
        if (!t.valid) { s = &t; break; }
    if (!s) {   // evict round-robin; the old image may still be in use on some stream
        s = &c->slot[c->next];
        c->next = (c->next + 1) % kTableSlots;
        if (int rc = cuda_ok(cudaDeviceSynchronize(), "table cache eviction")) return rc;
        s->valid = false;
    }
    if (s->cap < floats) {
        if (s->dev) cudaFree(s->dev);
        if (s->pinned) cudaFreeHost(s->pinned);
        s->dev = s->pinned = nullptr;
        s->cap = 0;
        if (int rc = cuda_ok(cudaMalloc(&s->dev, floats * sizeof(float)), "cudaMalloc step table")) return rc;
        if (int rc = cuda_ok(cudaMallocHost(&s->pinned, floats * sizeof(float)), "cudaMallocHost step table")) return rc;
        s->cap = floats;
    }
    fill(s->pinned);
    if (int rc = cuda_ok(cudaMemcpyAsync(s->dev, s->pinned, floats * sizeof(float), cudaMemcpyHostToDevice, stream), "step table upload")) return rc;
    s->hash = hash;
    s->floats = floats;
    s->valid = true;
    *out = s->dev;
    return MMB_OK;
}

static uint64_t step_table_hash(const MmbStepTable* st, int T, bool with_sp) {
    const size_t n = (size_t)st->n_steps;
    uint64_t h = 0xCBF29CE484222325ull;
    h = hash_words(h, &st->n_steps, sizeof(st->n_steps));
    h = hash_words(h, &T, sizeof(T));
    h = hash_words(h, st->bc, n * sizeof(float));
    h = hash_words(h, st->cc, n * sizeof(float));
    if (with_sp && st->sp) h = hash_words(h, st->sp, n * sizeof(float));
    if (st->t) h = hash_words(h, st->t, n * sizeof(float));
    return hash_words(h, st->temb, n * T * sizeof(float));
}

static void fill_step_table(float* img, const MmbStepTable* st, int T) {
    const int n = st->n_steps;
    for (int i = 0; i < n; ++i) {
        img[(size_t)i * 4 + 0] = st->bc[i];
        img[(size_t)i * 4 + 1] = st->cc[i];
        img[(size_t)i * 4 + 2] = st->sp ? st->sp[i] : 0.0f;
        img[(size_t)i * 4 + 3] = st->t ? st->t[i] : 0.0f;
    }
    memcpy(img + (size_t)n * 4, st->temb, (size_t)n * T * sizeof(float));
}

}  // namespace mmb

using namespace mmb;

extern "C" {

int mmb_abi_version(void) { return MMB_ABI_VERSION; }

const char* mmb_last_error(void) { return g_error; }

size_t mmb_epic_packed_floats(const MmbEpicDims* dims) { return dims ? mmb_epic_layout(dims).total : 0; }

int mmb_epic_create(const MmbEpicDims* dims, const float* packed, size_t n_floats, int device, MmbEpicModel** out) {
    if (!dims || !packed || !out) return fail(MMB_EINVAL, "mmb_epic_create: null argument");
    const MmbEpicLayout lo = mmb_epic_layout(dims);
    if (n_floats != lo.total) return fail(MMB_EINVAL, "mmb_epic_create: blob has %zu floats, layout wants %zu", n_floats, lo.total);
    int prev = 0;
    if (int rc = cuda_ok(cudaGetDevice(&prev), "cudaGetDevice")) return rc;
    if (int rc = cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return rc;
    EpicModel* m = new (std::nothrow) EpicModel();
    if (!m) return fail(MMB_ENOMEM, "out of host memory");
    m->tables = table_cache_create();
    m->host_pipe = host_pipe_create();
    m->dims = *dims;
    m->layout = lo;
    m->device = device;
    m->w = nullptr;
    m->tc_image = nullptr;
    m->tc_image_bytes = 0;
    m->mma_image_f16 = nullptr;
    m->mma_image_f16_bytes = 0;
    m->wide = nullptr;
    int rc = cuda_ok(cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, device), "sm count");
    if (!rc) rc = cuda_ok(cudaMalloc(&m->w, lo.total * sizeof(float)), "cudaMalloc weights");
    if (!rc) rc = cuda_ok(cudaMemcpy(m->w, packed, lo.total * sizeof(float), cudaMemcpyHostToDevice), "weight upload");
    try {   // the one-time packing uses std::vector: nothing may throw across the C ABI
        if (!rc && tc_supported(dims, 128)) rc = tc_build_image(m, packed);
        if (!rc && mma_supported(dims, 64)) rc = mma_build_images(m, packed);
        if (!rc && wide_supported(dims, 128)) rc = wide_build_image(m, packed);
    } catch (...) {
        rc = fail(MMB_ENOMEM, "mmb_epic_create: out of host memory");
    }
    cudaSetDevice(prev);
    if (rc) {
        mmb_epic_destroy(reinterpret_cast<MmbEpicModel*>(m));
        return rc;
    }
    *out = reinterpret_cast<MmbEpicModel*>(m);
    return MMB_OK;
}

void mmb_epic_destroy(MmbEpicModel* handle) {
    EpicModel* m = reinterpret_cast<EpicModel*>(handle);
    if (!m) return;
    if (m->w) cudaFree(m->w);
    if (m->tc_image) cudaFree(m->tc_image);
    if (m->mma_image_f16) cudaFree(m->mma_image_f16);
    wide_free_image(m);
    table_cache_destroy(m->tables);
    host_pipe_destroy(m->host_pipe);
    delete m;
}

int mmb_epic_forward(const MmbEpicModel* handle, const float* x, const uint8_t* k, const uint8_t* mask,
                     const float* temb, int temb_stride, int B, int N,
                     float* v_out, float* logits_out, float* hidden_out, int precision, void* stream) {
    const EpicModel* m = reinterpret_cast<const EpicModel*>(handle);
    if (!m || !x || !k || !mask || !temb || !v_out || !logits_out) return fail(MMB_EINVAL, "mmb_epic_forward: null argument");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_epic_forward: negative size");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (precision == MMB_PREC_FP32)
        return launch_epic_forward_fp32(m, x, k, mask, temb, temb_stride, B, N, v_out, logits_out, hidden_out, s);
    if (precision == MMB_PREC_BF16) {
        if (m->wide && wide_supported(&m->dims, N))
            return launch_epic_forward_wide(m, x, k, mask, temb, temb_stride, B, N, v_out, logits_out, hidden_out, s);
        if (!m->tc_image || !tc_supported(&m->dims, N))
            return fail(MMB_EUNSUPPORTED, "tcgen05 trunks are built for H=16 (G<=32, no context features) and H=128 (G<=32), Dc=3, S<=8, N<=128; use fp32");
        return launch_epic_forward_tc(m, x, k, mask, temb, temb_stride, B, N, v_out, logits_out, hidden_out, s);
    }
    return fail(MMB_EINVAL, "unknown precision %d", precision);
}

int mmb_bridge_update(float* x, uint8_t* k, uint8_t* mask, const float* v, const float* logits,
                      const float* absorb_logit, const float* u_jump, const float* u_absorb,
                      float dt, float bc, float cc, float sp, int B, int N, int Dc, int S, int flags, void* stream) {
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_bridge_update: negative size");
    if (Dc < 1 || Dc > 8 || S < 1 || S > 32) return fail(MMB_EINVAL, "mmb_bridge_update: need 1<=Dc<=8, 1<=S<=32");
    if (!mask) return fail(MMB_EINVAL, "mmb_bridge_update: mask is null");
    if (!(flags & MMB_FLAG_NO_EULER) && (!x || !v)) return fail(MMB_EINVAL, "mmb_bridge_update: Euler step needs x and v");
    if (!(flags & MMB_FLAG_NO_JUMP) && (!k || !logits || !u_jump)) return fail(MMB_EINVAL, "mmb_bridge_update: jump needs k, logits, u_jump");
    if ((flags & MMB_FLAG_ABSORBING) && (!absorb_logit || !u_absorb)) return fail(MMB_EINVAL, "mmb_bridge_update: birth needs absorb_logit, u_absorb");
    const size_t P = (size_t)B * (size_t)N;
    if (P == 0) return MMB_OK;
    return launch_bridge_update(x, k, mask, v, logits, absorb_logit, u_jump, u_absorb, StepScalars{dt, bc, cc, sp},
                                P, Dc, S, flags, static_cast<cudaStream_t>(stream));
}

static size_t wide_generate_scratch_floats(const EpicModel* m, int B, int N);

size_t mmb_generate_workspace_bytes(const MmbEpicModel* handle, int B, int N, int precision) {
    const EpicModel* m = reinterpret_cast<const EpicModel*>(handle);
    (void)precision;
    if (!m) return 0;
    // the tensor-core paths' per-step time vectors (up to 4096 steps) and jet lists; the step table itself is cached on the handle
    const size_t a = tc_generate_scratch_floats(&m->dims, 4096, B), b = mma_generate_scratch_floats(&m->dims, 4096, B),
                 c = wide_generate_scratch_floats(m, B, N);
    return ((a > b ? a : b) > c ? (a > b ? a : b) : c) * sizeof(float);
}

// The 128-wide tcgen05 trunk has no fused loop: a solver step is its network evaluation (~0.2 ms per 1000 jets, epic_wide_tc.cu)
// followed by the HBM-bound update kernel on the heads it wrote, with this step's Philox draws.  Scratch (floats): heads v | logits |
// uniforms | context rows [B][T + X] (models with context features).
static size_t wide_generate_scratch_floats(const EpicModel* m, int B, int N) {
    if (!m->wide) return 0;
    const size_t P = (size_t)(B > 0 ? B : 0) * (N > 0 ? N : 0);
    return P * (m->dims.dim_continuous + m->dims.vocab_size + 1) + (size_t)(B > 0 ? B : 0) * (m->dims.dim_time_emb + m->dims.dim_context) + 16;
}

__global__ void wide_context_rows_kernel(const float* __restrict__ temb, const float* __restrict__ ctx, int B, int T, int X, float* __restrict__ rows) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * (T + X)) return;
    const int b = i / (T + X), c = i - b * (T + X);
    rows[i] = c < T ? temb[c] : ctx[(size_t)b * X + (c - T)];
}

static int generate_wide(const EpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* context, const MmbStepTable* st,
                         const float* table, const float* u_jump, uint64_t seed, uint64_t jet_offset, int B, int N, float* ws, cudaStream_t s) {
    const int Dc = m->dims.dim_continuous, S = m->dims.vocab_size, T = m->dims.dim_time_emb, X = m->dims.dim_context, n = st->n_steps;
    const size_t P = (size_t)B * N;
    float *v = ws, *logits = v + P * Dc, *rows = logits + P * S + P;
    for (int step = 0; step < n; ++step) {
        const float* temb = table + (size_t)n * 4 + (size_t)step * T;
        int stride = 0;
        if (X > 0) {
            wide_context_rows_kernel<<<(B * (T + X) + 255) / 256, 256, 0, s>>>(temb, context, B, T, X, rows);
            if (int rc = cuda_ok(cudaGetLastError(), "context rows launch")) return rc;
            temb = rows;
            stride = T + X;
        }
        if (int rc = launch_epic_forward_wide(m, x, k, mask, temb, stride, B, N, v, logits, nullptr, s)) return rc;
        const UpdateDraws draws{seed, jet_offset, step, N};   // Philox inside the update kernel unless uniforms were injected
        if (int rc = launch_bridge_update(x, k, const_cast<uint8_t*>(mask), v, logits, nullptr, u_jump ? u_jump + (size_t)step * P : nullptr, nullptr,
                                          StepScalars{st->dt, st->bc[step], st->cc[step], 0.0f}, P, Dc, S, MMB_FLAG_MULTIMODAL, s, &draws))
            return rc;
    }
    return MMB_OK;
}

int mmb_generate_supported(const MmbEpicModel* handle, int N, int precision) {
    const EpicModel* m = reinterpret_cast<const EpicModel*>(handle);
    if (!m || N < 1) return 0;
    if (precision == MMB_PREC_FP32) return 1;
    if (precision == MMB_PREC_BF16 && m->wide && wide_supported(&m->dims, N)) return 1;
    if (precision == MMB_PREC_BF16) return m->tc_image && tc_supported(&m->dims, N) && (m->dims.disc_head_hidden == 0 || m->dims.disc_head_hidden == m->dims.vocab_size);
    if (precision == MMB_PREC_F16) return m->mma_image_f16 && mma_supported(&m->dims, N);
    return 0;
}

static size_t generate_ws_floats(const EpicModel* m, int n_steps, int B, int N, int precision) {
    if (precision == MMB_PREC_BF16 && m->wide) return wide_generate_scratch_floats(m, B, N);
    return precision == MMB_PREC_F16 ? mma_generate_scratch_floats(&m->dims, n_steps, B) : tc_generate_scratch_floats(&m->dims, n_steps, B);
}

int mmb_generate(const MmbEpicModel* handle, float* x, uint8_t* k, const uint8_t* mask, const float* context,
                 const MmbStepTable* st, const float* u_jump, uint64_t seed, uint64_t jet_offset,
                 int B, int N, void* workspace, size_t workspace_bytes, int precision, void* stream) {
    const EpicModel* m = reinterpret_cast<const EpicModel*>(handle);
    if (!m || !x || !k || !mask || !st || !workspace) return fail(MMB_EINVAL, "mmb_generate: null argument");
    if (!st->temb || !st->bc || !st->cc) return fail(MMB_EINVAL, "mmb_generate: incomplete step table");
    if (B < 0 || N < 0 || st->n_steps < 0) return fail(MMB_EINVAL, "mmb_generate: negative size");
    if ((m->dims.dim_context > 0) != (context != nullptr))
        return fail(MMB_EINVAL, "mmb_generate: the model has %d context features, context pointer %s", m->dims.dim_context,
                    context ? "given" : "missing");
    const int T = m->dims.dim_time_emb, n = st->n_steps;
    if (workspace_bytes < generate_ws_floats(m, n, B, N, precision) * sizeof(float))
        return fail(MMB_ENOMEM, "mmb_generate: workspace %zu B too small for %d steps", workspace_bytes, n);
    if (B == 0 || N == 0 || n == 0) return MMB_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float* table = nullptr;   // device image, cached on the handle (no copy, no allocation once this table has been seen)
    try {
        if (int rc = table_cache_get(m->tables, step_table_hash(st, T, false), table_floats(n, T), s,
                                     [&](float* img) { fill_step_table(img, st, T); }, &table))
            return rc;
    } catch (...) {
        return fail(MMB_ENOMEM, "mmb_generate: host-side failure while caching the step table");
    }
    if (precision == MMB_PREC_FP32)
        return launch_generate_fp32(m, x, k, mask, context, table, n, st->dt, u_jump, seed, jet_offset, B, N, s);
    if (precision == MMB_PREC_BF16 && m->wide && wide_supported(&m->dims, N)) {
        return generate_wide(m, x, k, mask, context, st, table, u_jump, seed, jet_offset, B, N, static_cast<float*>(workspace), s);
    }
    if (precision == MMB_PREC_BF16) {
        if (!m->tc_image || !tc_supported(&m->dims, N))
            return fail(MMB_EUNSUPPORTED, "tcgen05 path is built for H=16, G<=32, Dc+S<=16, head<=16, N<=128; use fp32");
        return launch_generate_tc(m, x, k, mask, table, static_cast<float*>(workspace), n, st->dt, u_jump, seed, jet_offset, B, N, s);
    }
    if (precision == MMB_PREC_F16) {
        if (!m->mma_image_f16 || !mma_supported(&m->dims, N))
            return fail(MMB_EUNSUPPORTED, "warp-MMA engine is built for H=16, G<=32, Dc=3, S in {4,8}, head in {0,S}, N<=256; use fp32");
        return launch_generate_mma(m, x, k, mask, context, table, static_cast<float*>(workspace), n, st->dt, u_jump, seed, jet_offset, B, N, s);
    }
    return fail(MMB_EINVAL, "unknown precision %d", precision);
}

// per-chunk device buffers of mmb_generate_host, each rounded up to 256 B: x f32 | k int64 | mask int64 | k u8 | mask u8 | scratch
struct HostChunkLayout {
    size_t x, k64, m64, k8, m8, ctx, scratch, total;
    HostChunkLayout(const EpicModel* m, int Bc, int N, int n_steps, int precision) {
        const size_t P = (size_t)Bc * N;
        size_t at = 0;
        auto take = [&](size_t bytes) { const size_t o = at; at += (bytes + 255) & ~(size_t)255; return o; };
        x = take(P * m->dims.dim_continuous * sizeof(float));
        k64 = take(P * 8); m64 = take(P * 8); k8 = take(P); m8 = take(P);
        ctx = take((size_t)Bc * m->dims.dim_context * sizeof(float));
        scratch = take(generate_ws_floats(m, n_steps, Bc, N, precision) * sizeof(float));
        total = at;
    }
};

static int host_chunks(int B, int n_chunks) {
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > kHostMaxChunks) n_chunks = kHostMaxChunks;
    return n_chunks > B ? (B > 0 ? B : 1) : n_chunks;
}

// direct mode (n_chunks <= 0): flag | mask int64 | mask u8 | token int64 (range check only) | context | scratch
struct HostDirectLayout {
    size_t m64, m8, k64, ctx, scratch, total;
    HostDirectLayout(const EpicModel* m, int B, int N, int n_steps) {
        const size_t P = (size_t)B * N;
        size_t at = 256;
        auto take = [&](size_t bytes) { const size_t o = at; at += (bytes + 255) & ~(size_t)255; return o; };
        m64 = take(P * 8); m8 = take(P); k64 = take(P * 8);
        ctx = take((size_t)B * m->dims.dim_context * sizeof(float));
        scratch = take(mma_generate_scratch_floats(&m->dims, n_steps, B) * sizeof(float));
        total = at;
    }
};
constexpr int kFallbackChunks = 2;   // direct mode asked for, but a buffer is not page-locked or the engine is not the warp-MMA one

static size_t host_ws_chunked(const EpicModel* m, int B, int N, int n_steps, int n_chunks, int precision) {
    n_chunks = host_chunks(B, n_chunks);
    const int Bc = (B + n_chunks - 1) / n_chunks;
    return 256 + (size_t)n_chunks * HostChunkLayout(m, Bc, N, n_steps, precision).total;
}

size_t mmb_generate_host_workspace_bytes(const MmbEpicModel* handle, int B, int N, int n_steps, int n_chunks, int precision) {
    const EpicModel* m = reinterpret_cast<const EpicModel*>(handle);
    if (!m || B < 0 || N < 0 || n_steps < 0) return 0;
    if (n_chunks > 0) return host_ws_chunked(m, B, N, n_steps, n_chunks, precision);
    const size_t a = HostDirectLayout(m, B, N, n_steps).total, b = host_ws_chunked(m, B, N, n_steps, kFallbackChunks, precision);
    return a > b ? a : b;
}

// device-visible address of a page-locked host buffer, or null
static void* mapped_host_pointer(const void* host) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

int mmb_generate_host(const MmbEpicModel* handle, const float* x_in, const int64_t* k_in, const int64_t* mask_in,
                      const float* context_in, const MmbStepTable* st, uint64_t seed, uint64_t jet_offset, int B, int N,
                      float* x_out, int64_t* k_out, int32_t* bad_tokens, void* workspace, size_t workspace_bytes,
                      int n_chunks, int precision, void* stream) {
    const EpicModel* m = reinterpret_cast<const EpicModel*>(handle);
    if (!m || !x_in || !k_in || !mask_in || !st || !x_out || !k_out || !bad_tokens || !workspace)
        return fail(MMB_EINVAL, "mmb_generate_host: null argument");
    if (B < 0 || N < 0 || st->n_steps < 0) return fail(MMB_EINVAL, "mmb_generate_host: negative size");
    const int X = m->dims.dim_context;
    if ((X > 0) != (context_in != nullptr))
        return fail(MMB_EINVAL, "mmb_generate_host: the model has %d context features, context pointer %s", X, context_in ? "given" : "missing");
    if (workspace_bytes < mmb_generate_host_workspace_bytes(handle, B, N, st->n_steps, n_chunks, precision))
        return fail(MMB_ENOMEM, "mmb_generate_host: workspace too small");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return fail(MMB_EINVAL, "mmb_generate_host: workspace must be 256-byte aligned");
    *bad_tokens = 0;
    if (B == 0 || N == 0 || st->n_steps == 0) return MMB_OK;
    HostPipe* hp = m->host_pipe;
    if (!hp) return fail(MMB_ENOMEM, "mmb_generate_host: no pipeline state");
    try {
        if (int rc = host_pipe_init(hp)) return rc;
    } catch (...) {
        return fail(MMB_ENOMEM, "mmb_generate_host: host-side failure");
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int S = m->dims.vocab_size;
    if (n_chunks <= 0) {
        // ---- direct mode: the warp-MMA kernel reads each jet's features and tokens from the mapped host buffers when a warp
        // claims it and writes the result straight back; only the masks (needed up front to bin the jets) and a copy of the
        // tokens for the range assertion travel by DMA, on two streams, under the kernel
        void *dx_in = mapped_host_pointer(x_in), *dk_in = mapped_host_pointer(k_in), *dx_out = mapped_host_pointer(x_out),
             *dk_out = mapped_host_pointer(k_out);
        const bool direct = precision == MMB_PREC_F16 && dx_in && dk_in && dx_out && dk_out && m->mma_image_f16 && mma_supported(&m->dims, N);
        if (direct) {
            const HostDirectLayout lay(m, B, N, st->n_steps);
            uint8_t* ws = static_cast<uint8_t*>(workspace);
            int* d_bad = reinterpret_cast<int*>(ws);
            const size_t P = (size_t)B * N;
            const int T = m->dims.dim_time_emb, n = st->n_steps;
            const float* table = nullptr;
            try {
                if (int rc = table_cache_get(m->tables, step_table_hash(st, T, false), table_floats(n, T), s,
                                             [&](float* img) { fill_step_table(img, st, T); }, &table))
                    return rc;
            } catch (...) {
                return fail(MMB_ENOMEM, "mmb_generate_host: host-side failure while caching the step table");
            }
            cudaStream_t sa = hp->stream[0], sb = hp->stream[1];
            long long* dm64 = reinterpret_cast<long long*>(ws + lay.m64);
            long long* dk64 = reinterpret_cast<long long*>(ws + lay.k64);
            uint8_t* dm8 = ws + lay.m8;
            int rc = cuda_ok(cudaMemsetAsync(d_bad, 0, sizeof(int), s), "flag reset");
            if (!rc) rc = cuda_ok(cudaEventRecord(hp->fork, s), "fork");
            if (!rc) rc = cuda_ok(cudaStreamWaitEvent(sa, hp->fork, 0), "fork wait");
            if (!rc) rc = cuda_ok(cudaStreamWaitEvent(sb, hp->fork, 0), "fork wait");
            if (!rc) rc = cuda_ok(cudaMemcpyAsync(dm64, mask_in, P * 8, cudaMemcpyHostToDevice, sa), "H2D mask");
            if (!rc) {
                narrow_mask_kernel<<<(unsigned)((P / 2 + 256) / 256), 256, 0, sa>>>(dm64, dm8, P);
                rc = cuda_ok(cudaGetLastError(), "narrow launch");
            }
            const MmaHostIO io{static_cast<const float*>(dx_in), static_cast<const long long*>(dk_in), static_cast<float*>(dx_out),
                               static_cast<long long*>(dk_out), d_bad};
            float* dctx = X ? reinterpret_cast<float*>(ws + lay.ctx) : nullptr;
            if (!rc && X) rc = cuda_ok(cudaMemcpyAsync(dctx, context_in, (size_t)B * X * sizeof(float), cudaMemcpyHostToDevice, sa), "H2D context");
            if (!rc) rc = launch_generate_mma(m, nullptr, nullptr, dm8, dctx, table, reinterpret_cast<float*>(ws + lay.scratch), n, st->dt, nullptr, seed,
                                              jet_offset, B, N, sa, &io);
            if (!rc) rc = cuda_ok(cudaEventRecord(hp->done[0], sa), "direct done");
            if (!rc) rc = cuda_ok(cudaMemcpyAsync(dk64, k_in, P * 8, cudaMemcpyHostToDevice, sb), "H2D tokens");
            if (!rc) {
                check_tokens_kernel<<<(unsigned)((P / 2 + 256) / 256), 256, 0, sb>>>(dk64, P, S, d_bad);
                rc = cuda_ok(cudaGetLastError(), "token check launch");
            }
            if (!rc) rc = cuda_ok(cudaEventRecord(hp->done[1], sb), "check done");
            cudaStreamWaitEvent(s, hp->done[0], 0);
            cudaStreamWaitEvent(s, hp->done[1], 0);
            if (!rc) rc = cuda_ok(cudaMemcpyAsync(bad_tokens, d_bad, sizeof(int), cudaMemcpyDeviceToHost, s), "D2H flag");
            return rc;
        }
        n_chunks = kFallbackChunks;
    }
    n_chunks = host_chunks(B, n_chunks);
    const int Bc = (B + n_chunks - 1) / n_chunks, Dc = m->dims.dim_continuous;
    const HostChunkLayout lay(m, Bc, N, st->n_steps, precision);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    int* d_bad = reinterpret_cast<int*>(ws);
    // fork: the chunk streams start after everything the caller enqueued on `stream` (and after the flag is cleared)
    int rc = cuda_ok(cudaMemsetAsync(d_bad, 0, sizeof(int), s), "flag reset");
    if (!rc) rc = cuda_ok(cudaEventRecord(hp->fork, s), "fork");
    for (int c = 0; c < n_chunks && !rc; ++c) {
        const int lo = c * Bc, hi = lo + Bc < B ? lo + Bc : B;
        if (hi <= lo) { n_chunks = c; break; }
        const size_t P = (size_t)(hi - lo) * N, off = (size_t)lo * N;
        cudaStream_t cs = hp->stream[c % kHostStreams];
        uint8_t* base = ws + 256 + (size_t)c * lay.total;
        float* dx = reinterpret_cast<float*>(base + lay.x);
        long long* dk64 = reinterpret_cast<long long*>(base + lay.k64);
        long long* dm64 = reinterpret_cast<long long*>(base + lay.m64);
        uint8_t *dk8 = base + lay.k8, *dm8 = base + lay.m8;
        rc = cuda_ok(cudaStreamWaitEvent(cs, hp->fork, 0), "fork wait");
        if (!rc) rc = cuda_ok(cudaMemcpyAsync(dx, x_in + off * Dc, P * Dc * sizeof(float), cudaMemcpyHostToDevice, cs), "H2D x");
        if (!rc) rc = cuda_ok(cudaMemcpyAsync(dk64, k_in + off, P * 8, cudaMemcpyHostToDevice, cs), "H2D k");
        if (!rc) rc = cuda_ok(cudaMemcpyAsync(dm64, mask_in + off, P * 8, cudaMemcpyHostToDevice, cs), "H2D mask");
        if (!rc) {
            narrow_state_kernel<<<(unsigned)((P / 2 + 256) / 256), 256, 0, cs>>>(dk64, dm64, dk8, dm8, P, S, d_bad);
            rc = cuda_ok(cudaGetLastError(), "narrow launch");
        }
        float* dctx = X ? reinterpret_cast<float*>(base + lay.ctx) : nullptr;
        if (!rc && X)
            rc = cuda_ok(cudaMemcpyAsync(dctx, context_in + (size_t)lo * X, (size_t)(hi - lo) * X * sizeof(float), cudaMemcpyHostToDevice, cs), "H2D context");
        if (!rc) rc = mmb_generate(handle, dx, dk8, dm8, dctx, st, nullptr, seed, jet_offset + (uint64_t)lo, hi - lo, N, base + lay.scratch,
                                   lay.total - lay.scratch, precision, cs);
        if (!rc) {
            widen_tokens_kernel<<<(unsigned)((P / 2 + 256) / 256), 256, 0, cs>>>(dk8, dk64, P);
            rc = cuda_ok(cudaGetLastError(), "widen launch");
        }
        if (!rc) rc = cuda_ok(cudaMemcpyAsync(x_out + off * Dc, dx, P * Dc * sizeof(float), cudaMemcpyDeviceToHost, cs), "D2H x");
        if (!rc) rc = cuda_ok(cudaMemcpyAsync(k_out + off, dk64, P * 8, cudaMemcpyDeviceToHost, cs), "D2H k");
        if (!rc) rc = cuda_ok(cudaEventRecord(hp->done[c], cs), "chunk done");
    }
    // join: the caller's stream continues after every chunk; the range flag follows them
    for (int c = 0; c < n_chunks; ++c) cudaStreamWaitEvent(s, hp->done[c], 0);
    if (!rc) rc = cuda_ok(cudaMemcpyAsync(bad_tokens, d_bad, sizeof(int), cudaMemcpyDeviceToHost, s), "D2H flag");
    return rc;
}

int mmb_philox_uniforms(float* u, uint64_t seed, uint64_t jet_offset, int n_steps, int B, int N, void* stream) {
    if (!u || n_steps < 0 || B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_philox_uniforms: bad argument");
    return launch_philox_uniforms(u, seed, jet_offset, 0, 0, n_steps, B, N, static_cast<cudaStream_t>(stream));
}

int mmb_jump_variants(const float* logits, const uint8_t* k, const float* u, float dt, float bc, float cc, size_t P, int S,
                      uint8_t* out_exact, uint8_t* out_tc, uint8_t* out_mma, void* stream) {
    if (!logits || !k || !u || !out_exact || !out_tc || !out_mma) return fail(MMB_EINVAL, "mmb_jump_variants: null argument");
    return launch_jump_variants(logits, k, u, StepScalars{dt, bc, cc, 0.0f}, P, S, out_exact, out_tc, out_mma, static_cast<cudaStream_t>(stream));
}

int mmb_absorb_head_create(int hidden, int transformer_dim, int n_heads, int n_blocks, const float* packed, size_t n_floats,
                           int device, MmbAbsorbHead** out) {
    if (!packed || !out) return fail(MMB_EINVAL, "mmb_absorb_head_create: null argument");
    AbsorbHead* h = nullptr;
    try {   // the one-time packing uses std::vector: nothing may throw across the C ABI
        if (int rc = absorb_head_create(hidden, transformer_dim, n_heads, n_blocks, packed, n_floats, device, &h)) return rc;
    } catch (...) {
        return fail(MMB_ENOMEM, "mmb_absorb_head_create: out of host memory");
    }
    *out = reinterpret_cast<MmbAbsorbHead*>(h);
    return MMB_OK;
}

void mmb_absorb_head_destroy(MmbAbsorbHead* h) { absorb_head_destroy(reinterpret_cast<AbsorbHead*>(h)); }

size_t mmb_absorb_head_workspace_bytes(int B) { return B < 0 ? 0 : tf_pack_scratch_ints(B) * sizeof(int32_t); }

int mmb_absorb_head_forward(const MmbAbsorbHead* head, const float* hidden, const uint8_t* mask, const float* tbias,
                            int tbias_stride, int B, int N, float* logit_out, void* workspace, size_t workspace_bytes, void* stream) {
    if (!head || !hidden || !mask || !tbias || !logit_out) return fail(MMB_EINVAL, "mmb_absorb_head_forward: null argument");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_absorb_head_forward: negative size");
    if (workspace && workspace_bytes < mmb_absorb_head_workspace_bytes(B)) return fail(MMB_ENOMEM, "mmb_absorb_head_forward: workspace too small");
    return launch_absorb_head(reinterpret_cast<const AbsorbHead*>(head), hidden, mask, tbias, tbias_stride, B, N, logit_out,
                              static_cast<cudaStream_t>(stream), static_cast<int32_t*>(workspace), workspace ? workspace_bytes / sizeof(int32_t) : 0);
}

// workspace of mmb_generate_absorbing (floats): v | logits | hidden | a | uj | ua   (the step table and the time biases are
// cached on the trunk's handle)
static size_t absorbing_ws_floats(const EpicModel* m, const AbsorbHead* h, int B, int N, int n_steps) {
    (void)h; (void)n_steps;
    const size_t P = (size_t)B * N;
    return P * (m->dims.dim_continuous + m->dims.vocab_size + m->dims.dim_hidden_local + 3) + 64 + tf_pack_scratch_ints(B) + 16;
}

size_t mmb_generate_absorbing_workspace_bytes(const MmbEpicModel* model, const MmbAbsorbHead* head, int B, int N, int n_steps) {
    if (!model || !head || B < 0 || N < 0 || n_steps < 0) return 0;
    return absorbing_ws_floats(reinterpret_cast<const EpicModel*>(model), reinterpret_cast<const AbsorbHead*>(head), B, N, n_steps) * sizeof(float);
}

int mmb_generate_absorbing(const MmbEpicModel* model, const MmbAbsorbHead* head, float* x, uint8_t* k, uint8_t* mask,
                           const MmbStepTable* st, const float* tbias, const float* u_jump, const float* u_absorb,
                           uint64_t seed, uint64_t jet_offset, int B, int N, void* workspace, size_t workspace_bytes,
                           int precision, void* stream) {
    const EpicModel* m = reinterpret_cast<const EpicModel*>(model);
    const AbsorbHead* h = reinterpret_cast<const AbsorbHead*>(head);
    if (!m || !h || !x || !k || !mask || !st || !tbias || !workspace) return fail(MMB_EINVAL, "mmb_generate_absorbing: null argument");
    if (m->dims.dim_context != 0)   // AbsorbingGenerator.forward passes batch.context_* on (absorbing_flows.py:150-153); not built for this loop
        return fail(MMB_EUNSUPPORTED, "mmb_generate_absorbing: the trunk was built with %d context features; this loop has no context input", m->dims.dim_context);
    if (!st->temb || !st->bc || !st->cc || !st->sp) return fail(MMB_EINVAL, "mmb_generate_absorbing: step table needs temb, bc, cc, sp");
    if (B < 0 || N < 0 || st->n_steps < 0) return fail(MMB_EINVAL, "mmb_generate_absorbing: negative size");
    if (absorb_head_hidden(h) != m->dims.dim_hidden_local) return fail(MMB_EINVAL, "head expects hidden %d, trunk has %d", absorb_head_hidden(h), m->dims.dim_hidden_local);
    const int T = m->dims.dim_time_emb, n = st->n_steps, Dc = m->dims.dim_continuous, S = m->dims.vocab_size, H = m->dims.dim_hidden_local;
    const int nblk = absorb_head_blocks(h);
    if (workspace_bytes < absorbing_ws_floats(m, h, B, N, n) * sizeof(float)) return fail(MMB_ENOMEM, "mmb_generate_absorbing: workspace too small");
    if (B == 0 || N == 0 || n == 0) return MMB_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t P = (size_t)B * N, tf = table_floats(n, T), nb = (size_t)n * nblk * 128;
    const float* img = nullptr;
    try {
        uint64_t hsh = hash_words(step_table_hash(st, T, true), tbias, nb * sizeof(float));
        hsh = hash_words(hsh, &nblk, sizeof(nblk));
        if (int rc = table_cache_get(m->tables, hsh, tf + nb, s, [&](float* dst) {
                fill_step_table(dst, st, T);
                memcpy(dst + tf, tbias, nb * sizeof(float));
            }, &img))
            return rc;
    } catch (...) {
        return fail(MMB_ENOMEM, "mmb_generate_absorbing: host-side failure while caching the step table");
    }
    float* ws = static_cast<float*>(workspace);
    const float* temb_dev = img + (size_t)n * 4;
    const float* tb_dev = img + tf;
    float* v = ws;
    float* logits = v + P * Dc;
    float* hidden = logits + P * S;
    float* alog = hidden + P * H;
    float* uj = alog + P;
    float* ua = uj + P;
    int32_t* pack = reinterpret_cast<int32_t*>(ua + P + 16);
    for (int i = 0; i < n; ++i) {
        // heads from the OLD mask (absorbing_flows.py:270), then birth -> Euler -> jump with the new one (:271-273)
        int rc = mmb_epic_forward(model, x, k, mask, temb_dev + (size_t)i * T, 0, B, N, v, logits, hidden, precision, stream);
        if (!rc) rc = launch_absorb_head(h, hidden, mask, tb_dev + (size_t)i * nblk * 128, 0, B, N, alog, s, pack, tf_pack_scratch_ints(B));
        // injected uniforms, or Philox drawn inside the update kernel (no uniform ever travels through HBM)
        const float* pj = u_jump ? u_jump + (size_t)i * P : nullptr;
        const float* pa = u_absorb ? u_absorb + (size_t)i * P : nullptr;
        const UpdateDraws draws{seed, jet_offset, i, N};
        if (!rc) rc = launch_bridge_update(x, k, mask, v, logits, alog, pj, pa, StepScalars{st->dt, st->bc[i], st->cc[i], st->sp[i]},
                                           P, Dc, S, MMB_FLAG_ABSORBING, s, &draws);
        if (rc) return rc;
    }
    return MMB_OK;
}

int mmb_validation_histograms(const float* x, const uint8_t* k, const uint8_t* mask, int B, int N, int Dc, int S,
                              int bins, float lo, float hi, int max_mult, uint64_t* counts, void* stream) {
    if (!x || !k || !mask || !counts) return fail(MMB_EINVAL, "mmb_validation_histograms: null argument");
    if (B < 0 || N < 0 || Dc < 1 || S < 1 || bins < 1 || max_mult < 0 || !(hi > lo))
        return fail(MMB_EINVAL, "mmb_validation_histograms: bad shape or range");
    if ((size_t)(Dc * bins + S + max_mult + 1) * 4 > 48 * 1024) return fail(MMB_EINVAL, "mmb_validation_histograms: too many bins");
    if (B == 0 || N == 0) return MMB_OK;
    return launch_validation_histograms(x, k, mask, B, N, Dc, S, bins, lo, hi, max_mult,
                                        reinterpret_cast<unsigned long long*>(counts), static_cast<cudaStream_t>(stream));
}

int mmb_jet_observables(const float* x, const uint8_t* k, const uint8_t* mask, const float* mean, const float* std, int B, int N,
                        float* x_phys, int8_t* flavor_charge, float* jets, void* stream) {
    if (!x || !k || !mask) return fail(MMB_EINVAL, "mmb_jet_observables: null argument");
    if ((mean == nullptr) != (std == nullptr)) return fail(MMB_EINVAL, "mmb_jet_observables: mean and std go together");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_jet_observables: negative size");
    if (B == 0 || N == 0) return MMB_OK;
    return launch_jet_observables(x, k, mask, mean, std, B, N, x_phys, flavor_charge, jets, static_cast<cudaStream_t>(stream));
}

int mmb_jet_substructure(const float* x, const uint8_t* mask, const float* mean, const float* std, int B, int N, float R, float beta,
                         float* out, int16_t* axes, void* stream) {
    if (!x || !mask || !out) return fail(MMB_EINVAL, "mmb_jet_substructure: null argument");
    if ((mean == nullptr) != (std == nullptr)) return fail(MMB_EINVAL, "mmb_jet_substructure: mean and std go together");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_jet_substructure: negative size");
    if (N > MMB_SUB_MAX_N) return fail(MMB_EINVAL, "mmb_jet_substructure: N = %d exceeds %d particle slots", N, MMB_SUB_MAX_N);
    if (!(R > 0.0f) || !(beta > 0.0f)) return fail(MMB_EINVAL, "mmb_jet_substructure: R and beta must be positive");
    if (B == 0) return MMB_OK;
    return launch_jet_substructure(x, mask, mean, std, B, N, R, beta, out, axes, static_cast<cudaStream_t>(stream));
}

int mmb_sample_source(float* x, uint8_t* k, uint8_t* mask, int B, int N, float scale, const float* cat_probs, const float* mult_cdf,
                      uint64_t seed, uint64_t jet_offset, void* stream) {
    if (!x || !k || !mask || !cat_probs) return fail(MMB_EINVAL, "mmb_sample_source: null argument");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_sample_source: negative size");
    if (B == 0 || N == 0) return MMB_OK;
    return launch_sample_source(x, k, mask, B, N, scale, cat_probs, mult_cdf, seed, jet_offset, static_cast<cudaStream_t>(stream));
}

int mmb_sample_bridges(const float* x0, const float* x1, const uint8_t* k0, const uint8_t* k1, const float* t, float sigma, float gamma,
                       int S, const float* z, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N, float* xt, uint8_t* kt,
                       void* stream) {
    if (!x0 || !x1 || !k0 || !k1 || !t || !xt || !kt) return fail(MMB_EINVAL, "mmb_sample_bridges: null argument");
    if ((z == nullptr) != (u == nullptr)) return fail(MMB_EINVAL, "mmb_sample_bridges: inject z and u together or neither");
    if (B < 0 || N < 0 || S < 1 || S > 255) return fail(MMB_EINVAL, "mmb_sample_bridges: bad size");
    if (B == 0 || N == 0) return MMB_OK;
    return launch_sample_bridges(x0, x1, k0, k1, t, sigma, gamma, S, z, u, seed, jet_offset, B, N, xt, kt, static_cast<cudaStream_t>(stream));
}

int mmb_absorbing_sample(const float* sp, const uint8_t* target_mask, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N,
                         uint8_t* mask_t, void* stream) {
    if (!sp || !target_mask || !mask_t) return fail(MMB_EINVAL, "mmb_absorbing_sample: null argument");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_absorbing_sample: negative size");
    if (B == 0 || N == 0) return MMB_OK;
    return launch_absorbing_sample(sp, target_mask, u, seed, jet_offset, B, N, mask_t, static_cast<cudaStream_t>(stream));
}

size_t mmb_bridge_losses_workspace_bytes(int B, int N) {
    if (B < 0 || N < 0) return 0;
    return (size_t)bridge_losses_blocks((size_t)B * N) * 3 * sizeof(float);
}

int mmb_bridge_losses(const float* v, const float* logits, const float* x0, const float* x1, const uint8_t* k1, const uint8_t* mask,
                      int B, int N, int S, float* out, void* workspace, size_t workspace_bytes, void* stream) {
    if (!v || !logits || !x0 || !x1 || !k1 || !mask || !out || !workspace) return fail(MMB_EINVAL, "mmb_bridge_losses: null argument");
    if (B < 1 || N < 1 || S < 1) return fail(MMB_EINVAL, "mmb_bridge_losses: bad size");
    if (workspace_bytes < mmb_bridge_losses_workspace_bytes(B, N)) return fail(MMB_ENOMEM, "mmb_bridge_losses: workspace too small");
    return launch_bridge_losses(v, logits, x0, x1, k1, mask, (size_t)B * N, S, out, static_cast<float*>(workspace),
                                static_cast<cudaStream_t>(stream));
}

static int check_grad_shape(const MmbEpicDims* d, int B, int N) {
    if (!d) return fail(MMB_EINVAL, "mmb_epic_loss_grad: null dims");
    if (d->dim_continuous < 1 || d->dim_continuous > 8 || d->vocab_size < 1 || d->vocab_size > 32)
        return fail(MMB_EINVAL, "mmb_epic_loss_grad: need 1 <= Dc <= 8 and 1 <= S <= 32 (got Dc=%d S=%d)", d->dim_continuous, d->vocab_size);
    if (d->dim_hidden_local < 1 || d->dim_hidden_glob < 1 || d->dim_time_emb < 1 || d->dim_cont_emb < 0 || d->dim_disc_emb < 0 ||
        d->num_blocks < 0 || d->dim_context < 0 || d->disc_head_hidden < 0)
        return fail(MMB_EINVAL, "mmb_epic_loss_grad: bad EPiC widths");
    if (B < 1 || N < 1 || N > MMB_EPIC_GRAD_MAX_N)
        return fail(MMB_EINVAL, "mmb_epic_loss_grad: need B >= 1 and 1 <= N <= %d (got B=%d N=%d)", MMB_EPIC_GRAD_MAX_N, B, N);
    return MMB_OK;
}

size_t mmb_epic_loss_grad_workspace_bytes(const MmbEpicDims* dims, int B, int N) {
    if (check_grad_shape(dims, B, N)) return 0;
    return epic_loss_grad_workspace_bytes(*dims, B, N);
}

int mmb_epic_loss_grad(const MmbEpicDims* dims, const float* W, const float* x, const uint8_t* k, const uint8_t* mask, const float* temb,
                       int temb_stride, const float* x0, const float* x1, const uint8_t* k1, int B, int N, float* losses, float* jac,
                       float* d_context, void* workspace, size_t workspace_bytes, void* stream) {
    if (int rc = check_grad_shape(dims, B, N)) return rc;
    if (!W || !x || !k || !mask || !temb || !x0 || !x1 || !k1 || !losses || !workspace)
        return fail(MMB_EINVAL, "mmb_epic_loss_grad: null argument");
    if (temb_stride < 0) return fail(MMB_EINVAL, "mmb_epic_loss_grad: negative temb_stride");
    const size_t need = epic_loss_grad_workspace_bytes(*dims, B, N);
    if (workspace_bytes < need) return fail(MMB_ENOMEM, "mmb_epic_loss_grad: workspace has %zu B, needs %zu B", workspace_bytes, need);
    return launch_epic_loss_grad(*dims, W, x, k, mask, temb, temb_stride, x0, x1, k1, B, N, losses, jac, d_context, workspace,
                                 static_cast<cudaStream_t>(stream));
}

size_t mmb_wasserstein1d_workspace_bytes(int n, int m, int K) {
    if (n < 0 || m < 0 || K < 1 || K > MMB_W1_MAX_K) return 0;
    return wasserstein1d_workspace_bytes(n, m, K);
}

int mmb_wasserstein1d(const float* x, int64_t ldx, int n, const float* y, int64_t ldy, int m, int K,
                      double* out, int64_t* n_used, void* workspace, size_t workspace_bytes, void* stream) {
    if (K < 1 || K > MMB_W1_MAX_K) return fail(MMB_EINVAL, "mmb_wasserstein1d: K = %d outside 1..%d", K, MMB_W1_MAX_K);
    if (n < 0 || m < 0) return fail(MMB_EINVAL, "mmb_wasserstein1d: negative size");
    if (ldx < K || ldy < K) return fail(MMB_EINVAL, "mmb_wasserstein1d: row strides must be >= K = %d", K);
    if ((!x && n > 0) || (!y && m > 0) || !out || !workspace) return fail(MMB_EINVAL, "mmb_wasserstein1d: null argument");
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(MMB_EINVAL, "mmb_wasserstein1d: workspace not 256-byte aligned");
    const size_t need = wasserstein1d_workspace_bytes(n, m, K);
    if (need == 0) return MMB_ECUDA;   // the size query failed and set the error text
    if (workspace_bytes < need) return fail(MMB_ENOMEM, "mmb_wasserstein1d: workspace %zu B, needs %zu B", workspace_bytes, need);
    return launch_wasserstein1d(x, ldx, n, y, ldy, m, K, out, reinterpret_cast<long long*>(n_used), workspace,
                                static_cast<cudaStream_t>(stream));
}

static bool drawn_sizes_ok(int draws, int rows, int P, int F) {
    return F >= 1 && F <= MMB_W1_MAX_K && P >= 1 && draws >= 1 && rows >= 1 && (long long)rows * P <= 0x7FFFFFFFLL &&
           2LL * draws * F <= 0x7FFFFFFFLL;   // segments (sample, draw, feature) are counted in int
}

size_t mmb_wasserstein1d_drawn_workspace_bytes(int draws, int rows, int P, int F) {
    return drawn_sizes_ok(draws, rows, P, F) ? wasserstein1d_drawn_workspace_bytes(draws, rows, P, F) : 0;
}

static bool drawn_strides_ok(int64_t ld_jet, int64_t ld_slot, const uint8_t* mask, int64_t ldm, int P, int F) {
    return (P == 1 || ld_slot >= F) && ld_jet >= (int64_t)(P - 1) * ld_slot + F && (!mask || ldm >= P);
}

int mmb_wasserstein1d_drawn(const float* x, int64_t ldx_jet, int64_t ldx_slot, const uint8_t* mask_x, int64_t ldmx, int n,
                            const float* y, int64_t ldy_jet, int64_t ldy_slot, const uint8_t* mask_y, int64_t ldmy, int m,
                            int P, int F, const int32_t* idx_x, const int32_t* idx_y, int draws, int rows,
                            double* out, int64_t* n_used, void* workspace, size_t workspace_bytes, void* stream) {
    if (!drawn_sizes_ok(draws, rows, P, F))
        return fail(MMB_EINVAL, "mmb_wasserstein1d_drawn: draws = %d, rows = %d, P = %d, F = %d (need >= 1, >= 1, rows * P and 2 * draws * F <= 2^31 - 1, F in 1..%d)",
                    draws, rows, P, F, MMB_W1_MAX_K);
    if (n < 1 || m < 1) return fail(MMB_EINVAL, "mmb_wasserstein1d_drawn: n and m must be positive");
    if (!drawn_strides_ok(ldx_jet, ldx_slot, mask_x, ldmx, P, F) || !drawn_strides_ok(ldy_jet, ldy_slot, mask_y, ldmy, P, F))
        return fail(MMB_EINVAL, "mmb_wasserstein1d_drawn: strides overlap for P = %d, F = %d", P, F);
    if (!x || !y || !idx_x || !idx_y || !out || !workspace) return fail(MMB_EINVAL, "mmb_wasserstein1d_drawn: null argument");
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(MMB_EINVAL, "mmb_wasserstein1d_drawn: workspace not 256-byte aligned");
    const size_t need = wasserstein1d_drawn_workspace_bytes(draws, rows, P, F);
    if (need == 0) return MMB_ECUDA;   // a size query failed and set the error text
    if (workspace_bytes < need) return fail(MMB_ENOMEM, "mmb_wasserstein1d_drawn: workspace %zu B, needs %zu B", workspace_bytes, need);
    return launch_wasserstein1d_drawn(x, ldx_jet, ldx_slot, mask_x, ldmx, y, ldy_jet, ldy_slot, mask_y, ldmy, P, F, idx_x, idx_y, draws, rows,
                                      out, reinterpret_cast<long long*>(n_used), workspace, static_cast<cudaStream_t>(stream));
}

int mmb_energy_flow_polynomials(const float* x, const uint8_t* mask, const float* mean, const float* std, int B, int N, float beta,
                                float* out, void* stream) {
    if (!x || !mask || !out) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials: null argument");
    if ((mean == nullptr) != (std == nullptr)) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials: mean and std go together");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials: negative size");
    if (N > MMB_SUB_MAX_N) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials: N = %d exceeds %d particle slots", N, MMB_SUB_MAX_N);
    if (!(beta > 0.0f)) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials: beta must be positive");
    if (B == 0) return MMB_OK;
    return launch_energy_flow_polynomials(x, mask, mean, std, B, N, beta, out, static_cast<cudaStream_t>(stream));
}

int mmb_energy_flow_polynomials_d4(const float* x, const uint8_t* mask, const float* mean, const float* std, int B, int N,
                                   float beta, float* out, void* stream) {
    if (!x || !mask || !out) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials_d4: null argument");
    if ((mean == nullptr) != (std == nullptr)) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials_d4: mean and std go together");
    if (B < 0 || N < 0) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials_d4: negative size");
    if (N > MMB_SUB_MAX_N)
        return fail(MMB_EINVAL, "mmb_energy_flow_polynomials_d4: N = %d exceeds %d particle slots", N, MMB_SUB_MAX_N);
    if (!(beta > 0.0f)) return fail(MMB_EINVAL, "mmb_energy_flow_polynomials_d4: beta must be positive");
    if (B == 0) return MMB_OK;
    return launch_energy_flow_polynomials_d4(x, mask, mean, std, B, N, beta, out, static_cast<cudaStream_t>(stream));
}

int mmb_sampled_moments(const float* x, int64_t ldx, int n, int d, const float* scale, const int32_t* idx, int draws, int rows,
                        double* sum, double* sumsq, void* stream) {
    if (d < 1 || d > MMB_MET_MAX_D) return fail(MMB_EINVAL, "mmb_sampled_moments: d = %d outside 1..%d", d, MMB_MET_MAX_D);
    if (n < 1 || draws < 1 || rows < 1) return fail(MMB_EINVAL, "mmb_sampled_moments: n, draws and rows must be positive");
    if (ldx < d) return fail(MMB_EINVAL, "mmb_sampled_moments: row stride must be >= d = %d", d);
    if (!x || !idx || !sum || !sumsq) return fail(MMB_EINVAL, "mmb_sampled_moments: null argument");
    return launch_sampled_moments(x, ldx, d, scale, idx, draws, rows, sum, sumsq, static_cast<cudaStream_t>(stream));
}

static bool kpd_sizes_ok(int batches, int B, int d) { return batches >= 1 && batches <= 65535 && B >= 2 && d >= 1 && d <= MMB_MET_MAX_D; }

size_t mmb_kpd_mmd_workspace_bytes(int batches, int B, int d) {
    return kpd_sizes_ok(batches, B, d) ? kpd_mmd_workspace_bytes(batches, B, d) : 0;
}

int mmb_kpd_mmd(const float* real, int64_t ldr, int n, const float* gen, int64_t ldg, int m, int d, const float* scale,
                const int32_t* idx_real, const int32_t* idx_gen, int batches, int B, int degree, double* out, void* workspace,
                size_t workspace_bytes, void* stream) {
    if (!kpd_sizes_ok(batches, B, d))
        return fail(MMB_EINVAL, "mmb_kpd_mmd: batches = %d, B = %d, d = %d (need 1..65535, >= 2, 1..%d)", batches, B, d, MMB_MET_MAX_D);
    if (n < 1 || m < 1 || degree < 1) return fail(MMB_EINVAL, "mmb_kpd_mmd: n, m and degree must be positive");
    if (ldr < d || ldg < d) return fail(MMB_EINVAL, "mmb_kpd_mmd: row strides must be >= d = %d", d);
    if (!real || !gen || !idx_real || !idx_gen || !out || !workspace) return fail(MMB_EINVAL, "mmb_kpd_mmd: null argument");
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(MMB_EINVAL, "mmb_kpd_mmd: workspace not 256-byte aligned");
    const size_t need = kpd_mmd_workspace_bytes(batches, B, d);
    if (workspace_bytes < need) return fail(MMB_ENOMEM, "mmb_kpd_mmd: workspace %zu B, needs %zu B", workspace_bytes, need);
    return launch_kpd_mmd(real, ldr, gen, ldg, d, scale, idx_real, idx_gen, batches, B, degree, out, workspace,
                          static_cast<cudaStream_t>(stream));
}

}  // extern "C"
