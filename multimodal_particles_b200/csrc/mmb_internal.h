// mmb_internal.h — declarations shared between the translation units of libmmbridge.so.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/mmbridge.h"

namespace mmb {

struct StepScalars;

// error plumbing (api.cu): records the message for mmb_last_error() and returns the code
int fail(int code, const char* fmt, ...);
int cuda_ok(cudaError_t e, const char* what);

// Device-resident model: the packed fp32 blob (layout of include/mmbridge.h) plus the operand
// images the tcgen05 path consumes.
// Device copies of the per-step host tables (MmbStepTable rows, absorbing time biases), cached on the model handle and
// keyed by a hash of their content: the first call with a table uploads it through a page-locked staging buffer on the
// caller's stream, later calls neither copy nor allocate (api.cu).
struct TableCache;
TableCache* table_cache_create();
void table_cache_destroy(TableCache* c);

struct HostPipe;   // streams / events of mmb_generate_host (api.cu)

struct EpicModel {
    TableCache* tables;
    HostPipe* host_pipe;
    MmbEpicDims dims;
    MmbEpicLayout layout;
    int device;
    int sm_count;
    float* w;             // [layout.total] fp32, device
    void* tc_image;       // bf16 UMMA operand image + fp32 side tables (epic_tc.cu), device; may be null
    size_t tc_image_bytes;
    void* mma_image_f16;  // B-fragment tiles of the warp-MMA engine (epic_mma.cu), fp16 operands; may be null
    size_t mma_image_f16_bytes;
    void* wide;           // operand image + tables of the 128-wide tcgen05 trunk (epic_wide_tc.cu); may be null
};

// bridge_update.cu
// uniforms drawn inside the update kernel (uj / ua null): the draws of solver step `step` for jets of N particle slots, keyed like
// mmb_philox_uniforms (stream 0 = jump, 1 = absorbing birth)
struct UpdateDraws {
    uint64_t seed, jet_offset;
    int step, N;
};
int launch_bridge_update(float* x, uint8_t* k, uint8_t* mask, const float* v, const float* logits,
                         const float* absorb, const float* uj, const float* ua, StepScalars sc,
                         size_t P, int Dc, int S, int flags, cudaStream_t stream, const UpdateDraws* draws = nullptr);
int launch_philox_uniforms(float* u, uint64_t seed, uint64_t jet_offset, int stream_id, int step0, int n_steps, int B, int N,
                           cudaStream_t stream);

int launch_jump_variants(const float* logits, const uint8_t* k, const float* u, StepScalars sc, size_t P, int S, uint8_t* out_exact,
                         uint8_t* out_tc, uint8_t* out_mma, cudaStream_t stream);

// absorb_head_tc.cu — 128-wide transformer stack (ResnetBlock + AttnBlock) on tcgen05
struct TfStack {
    int Cin = 0, n_blocks = 0, n_jet = 0;
    void* image = nullptr;    // bf16 operand tiles, one 36 KB slot per streamed matrix
    float* table = nullptr;   // fp32 side table (norm affine, biases, per-particle output vector)
    float* jet_wT = nullptr;  // [128][n_jet] per-jet head on the slot mean
    float* jet_b = nullptr;
};
struct TfStackIO {
    int mode;                 // 0: [hidden, one_hot(mask)]; 1: [hidden, onehot]; 2: mask * [hidden, onehot, dist, near, !near]
    int H, S;
    const float* hidden;      // [B,N,H]
    const uint8_t* mask;      // [B,N]
    const float* onehot;      // [B,N,S]  modes 1, 2
    const float* x;           // [B,N,3]  mode 2
    const int32_t* nearest;   // [B]      mode 2
    const float* tbias;       // [B or 1][n_blocks][128]
    int tbias_stride;
    float* dot_out;           // [B,N]
    float* jet_out;           // [B][128] means of X over the slots (input of launch_jet_head) or null
    int32_t* pack_scratch;    // tf_pack_scratch_ints(B) ints of device memory: the kernel then computes padded slots once and packs
    size_t pack_scratch_ints; // several jets into a tile; null = one jet per tile, one row per slot
};
size_t tf_pack_scratch_ints(int B);
int tf_stack_build(TfStack* st, const float* proj_in, int Cin, const float* blocks, int n_blocks, const float* dot_w, float dot_c,
                   const float* jet_w, const float* jet_b, int n_jet);
void tf_stack_free(TfStack* st);
int launch_tf_stack(const TfStack* st, int sm_count, const TfStackIO& io, int B, int N, cudaStream_t stream);
// out [B][n_jet] = folded per-jet Linear of the stack applied to the slot means written by launch_tf_stack
int launch_jet_head(const TfStack* st, const float* means, int B, float* out, cudaStream_t stream);

struct AbsorbHead;
int absorb_head_create(int H, int C, int n_heads, int n_blocks, const float* W, size_t n_floats, int device, AbsorbHead** out);
void absorb_head_destroy(AbsorbHead* h);
int absorb_head_hidden(const AbsorbHead* h);
int absorb_head_blocks(const AbsorbHead* h);
int launch_absorb_head(const AbsorbHead* h, const float* hidden, const uint8_t* mask, const float* tbias, int tbias_stride,
                       int B, int N, float* logit_out, cudaStream_t stream, int32_t* pack_scratch = nullptr, size_t pack_scratch_ints = 0);

// histograms.cu
int launch_validation_histograms(const float* x, const uint8_t* k, const uint8_t* mask, int B, int N, int Dc, int S,
                                 int bins, float lo, float hi, int max_mult, unsigned long long* counts, cudaStream_t stream);

int launch_jet_observables(const float* x, const uint8_t* k, const uint8_t* mask, const float* mean, const float* sd, int B, int N,
                           float* x_phys, int8_t* fc, float* jets, cudaStream_t stream);

// substructure.cu — N-subjettiness and energy correlation functions, one block per jet, N <= MMB_SUB_MAX_N
int launch_jet_substructure(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N, float R, float beta,
                            float* out, int16_t* axes, cudaStream_t stream);

// wasserstein.cu — per-column 1-D W1: key pre-pass, CUB radix sort per column, merge-path integration in fixed tiles
size_t wasserstein1d_workspace_bytes(int n, int m, int K);   // 0 when the CUB size query fails
int launch_wasserstein1d(const float* x, long long ldx, int n, const float* y, long long ldy, int m, int K, double* out, long long* n_used,
                         void* workspace, cudaStream_t stream);
// the same per draw and feature over the used slots of drawn jets: key expansion into segments of capacity rows * P, one sort each
size_t wasserstein1d_drawn_workspace_bytes(int draws, int rows, int P, int F);   // 0 when a CUB size query fails
int launch_wasserstein1d_drawn(const float* x, long long ldx_jet, long long ldx_slot, const uint8_t* mask_x, long long ldmx, const float* y,
                               long long ldy_jet, long long ldy_slot, const uint8_t* mask_y, long long ldmy, int P, int F, const int32_t* idx_x,
                               const int32_t* idx_y, int draws, int rows, double* out, long long* n_used, void* workspace,
                               cudaStream_t stream);

// efp.cu — energy flow polynomials, one block per jet, Theta as an upper triangle of 32 x 32 blocks in shared memory
int launch_energy_flow_polynomials(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N, float beta,
                                   float* out, cudaStream_t stream);
int launch_energy_flow_polynomials_d4(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N,
                                      float beta, float* out, cudaStream_t stream);

// jet_metrics.cu — FPD moments over drawn rows, KPD unbiased MMD^2 over row strips with fixed-order partials
int launch_sampled_moments(const float* x, long long ldx, int d, const float* scale, const int* idx, int draws, int rows, double* sum,
                           double* sumsq, cudaStream_t stream);
size_t kpd_mmd_workspace_bytes(int batches, int B, int d);
int launch_kpd_mmd(const float* real, long long ldr, const float* gen, long long ldg, int d, const float* scale, const int* idx_real,
                   const int* idx_gen, int batches, int B, int degree, double* out, void* workspace, cudaStream_t stream);

int launch_sample_source(float* x, uint8_t* k, uint8_t* mask, int B, int N, float scale, const float* cat_probs, const float* mult_cdf,
                         uint64_t seed, uint64_t jet_offset, cudaStream_t stream);

// bridge_sample.cu — forward half of a training / validation step
int launch_sample_bridges(const float* x0, const float* x1, const uint8_t* k0, const uint8_t* k1, const float* ts, float sigma, float gamma,
                          int S, const float* z, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N, float* xt, uint8_t* kt,
                          cudaStream_t stream);
int launch_absorbing_sample(const float* sp, const uint8_t* target_mask, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N,
                            uint8_t* mask_t, cudaStream_t stream);
int bridge_losses_blocks(size_t P);
int launch_bridge_losses(const float* v, const float* logits, const float* x0, const float* x1, const uint8_t* k1, const uint8_t* mask,
                         size_t P, int S, float* out, float* partial, cudaStream_t stream);

// epic_fp32.cu — CUDA-core path, bit-identical to the oracle
int launch_epic_forward_fp32(const EpicModel* m, const float* x, const uint8_t* k, const uint8_t* mask,
                             const float* temb, int temb_stride, int B, int N,
                             float* v_out, float* logits_out, float* hidden_out, cudaStream_t stream);
// device step table: [n_steps] rows of (bc, cc, sp, pad) followed by [n_steps][T] temb
int launch_generate_fp32(const EpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* context, const float* dev_table,
                         int n_steps, float dt, const float* u_jump, uint64_t seed, uint64_t jet_offset,
                         int B, int N, cudaStream_t stream);

// epic_grad.cu — bridge-matching losses and their weight gradients, fp32 (arguments checked by the caller)
size_t epic_loss_grad_workspace_bytes(const MmbEpicDims& d, int B, int N);
int launch_epic_loss_grad(const MmbEpicDims& d, const float* W, const float* x, const uint8_t* k, const uint8_t* mask, const float* temb,
                          int temb_stride, const float* x0, const float* x1, const uint8_t* k1, int B, int N, float* losses, float* jac,
                          float* d_context, void* workspace, cudaStream_t stream);

// epic_tc.cu — tcgen05 path
bool tc_supported(const MmbEpicDims* d, int N);
int tc_build_image(EpicModel* m, const float* packed_host);
int launch_epic_forward_tc(const EpicModel* m, const float* x, const uint8_t* k, const uint8_t* mask,
                           const float* temb, int temb_stride, int B, int N,
                           float* v_out, float* logits_out, float* hidden_out, cudaStream_t stream);
size_t tc_generate_scratch_floats(const MmbEpicDims* d, int n_steps, int B);
int launch_generate_tc(const EpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* dev_table, float* scratch,
                       int n_steps, float dt, const float* u_jump, uint64_t seed, uint64_t jet_offset,
                       int B, int N, cudaStream_t stream);

// epic_wide_tc.cu — tcgen05 trunk for dim_hidden_local = 128 (the reference's class default, epic.py:99-101)
bool wide_supported(const MmbEpicDims* d, int N);
int wide_build_image(EpicModel* m, const float* packed_host);
void wide_free_image(EpicModel* m);
int launch_epic_forward_wide(const EpicModel* m, const float* x, const uint8_t* k, const uint8_t* mask, const float* temb, int temb_stride,
                             int B, int N, float* v_out, float* logits_out, float* hidden_out, cudaStream_t stream);

// epic_mma.cu — warp-level MMA engine (register-resident chains), generation only
bool mma_supported(const MmbEpicDims* d, int N);
int mma_build_images(EpicModel* m, const float* packed_host);
size_t mma_generate_scratch_floats(const MmbEpicDims* d, int n_steps, int B);
struct MmaHostIO {          // direct mode of mmb_generate_host: device-visible addresses of the caller's page-locked host buffers
    const float* x_in;      // [B,N,Dc]
    const long long* k_in;  // [B,N] int64
    float* x_out;           // [B,N,Dc]
    long long* k_out;       // [B,N] int64
    int* bad_tokens;        // DEVICE flag
};
int launch_generate_mma(const EpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* context, const float* dev_table, float* scratch,
                        int n_steps, float dt, const float* u_jump, uint64_t seed, uint64_t jet_offset,
                        int B, int N, cudaStream_t stream, const MmaHostIO* host = nullptr);

}  // namespace mmb
