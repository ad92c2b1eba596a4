/*
 * mmbridge.h — C ABI of libmmbridge.so: the B200 (sm_100a) generation hot path of
 * Multimodal-Bridges (cesarali/multimodal_particles).
 *
 * The reference has no FFI: its hot path is a Python object API (SURVEY.md §8b).  Each entry
 * point below names the reference Python interface it stands behind (file:line under
 * /root/reference/multimodal_particles/, abbreviated mp/).  The binding a reference maintainer
 * would add is the ctypes stub shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer except `packed` in mmb_epic_create and the
 *     MmbStepTable arrays is a DEVICE pointer owned by the caller;
 *   - return 0 on success, a negative MMB_E* code otherwise; mmb_last_error() gives the text
 *     (thread-local); nothing throws across the ABI;
 *   - all compute calls are asynchronous on `stream` (a cudaStream_t passed as void*), make no
 *     hidden synchronisation and allocate nothing (workspace is sized by mmb_*_workspace_bytes
 *     and supplied by the caller);
 *   - tokens and masks are uint8 on the device ([B,N], values 0..S-1 and 0/1); the int64
 *     [B,N,1] layout of the reference (mp/models/generative/multimodal_bridge_matching.py:13-20)
 *     is narrowed/widened once per generation by the host shim.
 */
#ifndef MMBRIDGE_H
#define MMBRIDGE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMB_ABI_VERSION 3

enum {
    MMB_OK = 0,
    MMB_EINVAL = -1,       /* bad argument / unsupported shape */
    MMB_ECUDA = -2,        /* CUDA runtime error (text in mmb_last_error) */
    MMB_ENOMEM = -3,       /* workspace too small / shared memory limit */
    MMB_EUNSUPPORTED = -4  /* precision or config not built for this path */
};

/* flags for mmb_bridge_update / mmb_generate */
enum {
    MMB_FLAG_MULTIMODAL = 0, /* Euler + jump with the given mask      (mp/.../bridges.py:38-45,179-201) */
    MMB_FLAG_ABSORBING = 1,  /* birth step first: mask' = mask | born (mp/.../bridges.py:260-286), then used */
    MMB_FLAG_NO_EULER = 2,   /* leave x untouched  (a lone TelegraphBridge / AbsorbingBridge.solver_step) */
    MMB_FLAG_NO_JUMP = 4     /* leave k untouched  (a lone LinearUniformBridge / AbsorbingBridge.solver_step) */
};

/* arithmetic of the EPiC trunk */
enum {
    MMB_PREC_FP32 = 0, /* CUDA-core fp32, bit-identical to oracle/mmb_oracle.c */
    MMB_PREC_BF16 = 1, /* tcgen05 bf16 operands, fp32 accumulate in TMEM */
    MMB_PREC_F16 = 2   /* mmb_generate only: warp-level mma.sync chains held in registers, fp16 operands, fp32 accumulate */
};

/*
 * Shape of the EPiC encoder.  Mirrors the fields of EncoderConfig / JetsDataConfig that the
 * reference constructors read (mp/models/architectures/epic.py:20-58,
 * mp/config_classes/multimodal_bridge_matching_config.py:23-91).
 * Supported: SinusoidalPositionalEncoding time embedding, Linear continuous embedding,
 * Embedding discrete embedding.  Context features (epic.py:72-76, utils.py:155-170; zero in every shipped config): the
 * reference concatenates [time embedding | embedded continuous context | embedded discrete context] into one per-jet
 * `context` vector that enters global_0, fc_global1 and fc_local1.  dim_context is the width of the part after the time
 * embedding; the caller applies the (tiny, per-jet) context embeddings and hands over the embedded vector.
 */
typedef struct MmbEpicDims {
    int32_t dim_continuous;    /* Dc  data.dim_features_continuous */
    int32_t vocab_size;        /* S   data.vocab_size_features     */
    int32_t dim_time_emb;      /* T   encoder.dim_emb_time (= context width) */
    int32_t dim_cont_emb;      /* C   encoder.dim_emb_features_continuous */
    int32_t dim_disc_emb;      /* D   encoder.dim_emb_features_discrete   */
    int32_t dim_hidden_local;  /* H   encoder.dim_hidden_local */
    int32_t dim_hidden_glob;   /* G   encoder.dim_hidden_glob  */
    int32_t num_blocks;        /* L   encoder.num_blocks */
    int32_t skip_connection;   /* encoder.skip_connection */
    int32_t disc_head_hidden;  /* Sh: 0 = no discrete head; S for MultiModalEPiC.fc_layer
                                  (mp/.../multimodal_bridge_matching.py:90-100); 56 for
                                  AbsorbingGenerator.discrete_head_mlp (absorbing_flows.py:41-54) */
    int32_t dim_context;       /* X   dim_emb_context_continuous + dim_emb_context_discrete (0: no context features) */
} MmbEpicDims;

/*
 * Packed weight blob: fp32, weight-norm already folded (W = g * v / ||v||_row,
 * mp/models/architectures/epic.py:134,171-176,208-215), every matrix row-major [out][in],
 * each matrix followed by its bias, in this order (in-widths in brackets):
 *   emb_cont  [C][Dc] + [C]
 *   emb_disc  [S][D]                      (embedding table, no bias)
 *   proj.local_0  [H][T+C+D] + [H]
 *   proj.global_0 [H][2H+T+X] + [H]
 *   proj.global_1 [H][H]     + [H]
 *   proj.global_2 [G][H]     + [G]
 *   L x { fc_global1 [H][2H+G+T+X] + [H]; fc_global2 [G][H] + [G];
 *         fc_local1  [H][H+G+T+X]  + [H]; fc_local2  [H][H] + [H] }
 *   output_layer [Dc+S][H] + [Dc+S]
 *   if Sh: head0 [Sh][S] + [Sh]; head2 [S][Sh] + [S]
 */
typedef struct MmbEpicLayout {
    size_t emb_cont_w, emb_cont_b, emb_disc;
    size_t local0_w, local0_b, global0_w, global0_b, global1_w, global1_b, global2_w, global2_b;
    size_t layer0;       /* offset of the first EPiC layer */
    size_t layer_stride; /* floats per EPiC layer */
    size_t l_g1_w, l_g1_b, l_g2_w, l_g2_b, l_l1_w, l_l1_b, l_l2_w, l_l2_b; /* within a layer */
    size_t out_w, out_b, head0_w, head0_b, head2_w, head2_b;
    size_t total;
} MmbEpicLayout;

static inline MmbEpicLayout mmb_epic_layout(const MmbEpicDims* d) {
    MmbEpicLayout L;
    size_t o = 0;
    const size_t Dc = (size_t)d->dim_continuous, S = (size_t)d->vocab_size, T = (size_t)d->dim_time_emb,
                 C = (size_t)d->dim_cont_emb, D = (size_t)d->dim_disc_emb, H = (size_t)d->dim_hidden_local,
                 G = (size_t)d->dim_hidden_glob, Sh = (size_t)d->disc_head_hidden, X = (size_t)d->dim_context;
    L.emb_cont_w = o; o += C * Dc;
    L.emb_cont_b = o; o += C;
    L.emb_disc = o;   o += S * D;
    L.local0_w = o;   o += H * (T + C + D);
    L.local0_b = o;   o += H;
    L.global0_w = o;  o += H * (2 * H + T + X);
    L.global0_b = o;  o += H;
    L.global1_w = o;  o += H * H;
    L.global1_b = o;  o += H;
    L.global2_w = o;  o += G * H;
    L.global2_b = o;  o += G;
    L.layer0 = o;
    {
        size_t p = 0;
        L.l_g1_w = p; p += H * (2 * H + G + T + X);
        L.l_g1_b = p; p += H;
        L.l_g2_w = p; p += G * H;
        L.l_g2_b = p; p += G;
        L.l_l1_w = p; p += H * (H + G + T + X);
        L.l_l1_b = p; p += H;
        L.l_l2_w = p; p += H * H;
        L.l_l2_b = p; p += H;
        L.layer_stride = p;
    }
    o += L.layer_stride * (size_t)d->num_blocks;
    L.out_w = o; o += (Dc + S) * H;
    L.out_b = o; o += (Dc + S);
    L.head0_w = L.head0_b = L.head2_w = L.head2_b = 0;
    if (Sh) {
        L.head0_w = o; o += Sh * S;
        L.head0_b = o; o += Sh;
        L.head2_w = o; o += S * Sh;
        L.head2_b = o; o += S;
    }
    L.total = o;
    return L;
}

/*
 * Per-solver-step scalars, computed ON THE HOST with the reference's own fp32 op order so that no
 * libm-vs-libdevice difference enters (SURVEY.md §A.4):
 *   t      network time of the step            (mp/.../multimodal_bridge_matching.py:203-211)
 *   temb   [T] sinusoidal embedding of t        (mp/models/architectures/utils.py:183-198; T = dim_time_emb, no context part)
 *   bc,cc  telegraph coefficients B=(w S)/(1-w), C=w, w=exp(-S gamma (1-t))  (bridges.py:125-130)
 *   sp     absorbing survival probability SP(t) (bridges.py:218-231); unused for MULTIMODAL
 * Arrays are HOST pointers of length n_steps (temb: n_steps*T); mmb_generate copies nothing — it
 * reads them when launching each step.
 */
typedef struct MmbStepTable {
    int32_t n_steps;
    float dt;          /* (1-eps)/(T-1) as fp32 (mbm.py:209) */
    const float* t;
    const float* temb;
    const float* bc;
    const float* cc;
    const float* sp;   /* nullable */
} MmbStepTable;

typedef struct MmbEpicModel MmbEpicModel; /* opaque: device-resident weights in every layout the kernels use */

int mmb_abi_version(void);
const char* mmb_last_error(void);

/* number of floats mmb_epic_create expects for `dims` (== mmb_epic_layout(dims).total) */
size_t mmb_epic_packed_floats(const MmbEpicDims* dims);

/*
 * Build the device-side model from a HOST blob.  Stands behind the reference constructors
 * EPiCWrapper(config) + MultiModalEPiC.fc_layer (epic.py:20-58, mbm.py:80-100) and
 * load_state_dict of the keys listed in SURVEY.md §A.6.  Synchronous (one-time).
 */
int mmb_epic_create(const MmbEpicDims* dims, const float* packed, size_t n_floats, int device, MmbEpicModel** out);
void mmb_epic_destroy(MmbEpicModel* m);

/*
 * One network evaluation.  Stands behind MultiModalEPiC.forward (mbm.py:102-113) ==
 * EPiCWrapper.forward (epic.py:62-91) + the discrete head; with hidden_out != NULL it is
 * EPiCWrapper.forward(..., output_hidden_local=True) as AbsorbingGenerator.forward calls it
 * (absorbing_flows.py:153).
 *   x [B,N,Dc] f32, k [B,N] u8, mask [B,N] u8,
 *   temb [B,T+X] (temb_stride = T+X) or one row shared by all jets (temb_stride = 0): the time embedding followed,
 *   when the model has context features, by the jet's embedded context (the reference's `context` vector, utils.py:166-170),
 *   v_out [B,N,Dc], logits_out [B,N,S]; hidden_out [B,N,H] nullable.
 *   With context features MMB_PREC_FP32 only (MMB_PREC_BF16 returns MMB_EUNSUPPORTED).
 * An empty jet (mask all zero) produces NaN exactly as epic.py:141 does.
 */
int mmb_epic_forward(const MmbEpicModel* m, const float* x, const uint8_t* k, const uint8_t* mask,
                     const float* temb, int temb_stride, int B, int N,
                     float* v_out, float* logits_out, float* hidden_out,
                     int precision, void* stream);

/*
 * The fused hybrid update, in place.  Stands behind, in this order,
 *   AbsorbingBridge.solver_step      (bridges.py:260-286)   [ABSORBING only]
 *   LinearUniformBridge.solver_step  (bridges.py:38-45)
 *   TelegraphBridge.solver_step      (bridges.py:179-201) incl. .rate (bridges.py:106-132)
 * with the Poisson tau-leap replaced by its exactly equivalent one-uniform categorical
 * (SURVEY.md §A.4 Form B, self slot retained; DESIGN.md §3):
 *   x [B,N,Dc] f32 in/out, k [B,N] u8 in/out, mask [B,N] u8 (in; in/out for ABSORBING),
 *   v [B,N,Dc], logits [B,N,S], absorb_logit [B,N] (ABSORBING), u_jump [B,N], u_absorb [B,N].
 * Sub-steps are switched off with MMB_FLAG_NO_EULER / MMB_FLAG_NO_JUMP (their inputs may then be
 * NULL), which is how the host shim serves a lone bridge.solver_step call.
 * Returns MMB_EINVAL for S > 32 or Dc > 8.  Tokens outside [0,S) are undefined behaviour on the
 * device; the host shim keeps the reference's assertion (bridges.py:111-115).
 */
int mmb_bridge_update(float* x, uint8_t* k, uint8_t* mask,
                      const float* v, const float* logits, const float* absorb_logit,
                      const float* u_jump, const float* u_absorb,
                      float dt, float bc, float cc, float sp,
                      int B, int N, int Dc, int S, int flags, void* stream);

/*
 * Whole generation loop for the multimodal bridge: n_steps x (network, update) with the state
 * resident on the device.  Stands behind MultiModalBridgeMatching.simulate_dynamics
 * (mbm.py:199-216) minus the final .cpu().
 *   u_jump: [n_steps,B,N] pre-drawn uniforms, or NULL to draw in-kernel with Philox4x32-10 keyed by
 *   (seed, jet_offset + jet, step, particle) — results are then invariant to how jets are sharded.
 *   workspace: mmb_generate_workspace_bytes(m, B, N, precision) bytes of 16-byte aligned device memory (per-step time
 *   vectors and the jet lists of the tensor-core engines, which bin the jets of a call on the device — MMB_PREC_BF16: jets
 *   without a live particle at index >= 64 share a 128-row tile in pairs; MMB_PREC_F16: jets are claimed by warps in order of
 *   their width.  Where and when a jet runs depends on the jet alone, so results do not depend on the size or composition
 *   of the call either).  The device image of the step table is cached on the model handle: a call with a table the handle
 *   has seen neither copies nor allocates.
 *   An empty jet (mask all zero) ends with NaN features and zero tokens in every precision, as the reference's division by
 *   the particle count gives (epic.py:141, bridges.py:42).
 *   context: [B,X] f32 embedded context features of the jets (device; constant over the steps — batch.context_* of
 *   mbm.py:143-144 through the context embeddings), NULL iff the model has none (X = 0).  MMB_PREC_FP32 and MMB_PREC_F16.
 */
size_t mmb_generate_workspace_bytes(const MmbEpicModel* m, int B, int N, int precision);

/*
 * 1 if mmb_generate can run this model at N particles per jet in `precision`, else 0 (MMB_PREC_FP32 takes any shape; the
 * tensor-core engines are built for the default EPiC widths: hidden 16, G <= 32, Dc = 3, S in {4, 8}, head width 0 or S;
 * MMB_PREC_BF16: N <= 128, MMB_PREC_F16: N <= 256).  The host shim's precision "auto" asks in the order F16, BF16, FP32.
 */
int mmb_generate_supported(const MmbEpicModel* m, int N, int precision);
int mmb_generate(const MmbEpicModel* m, float* x, uint8_t* k, const uint8_t* mask, const float* context,
                 const MmbStepTable* steps, const float* u_jump,
                 uint64_t seed, uint64_t jet_offset, int B, int N,
                 void* workspace, size_t workspace_bytes, int precision, void* stream);

/*
 * The same generation with HOST buffers in the reference's own layout — what MultiModalBridgeMatching.simulate_dynamics
 * receives and returns (mbm.py:199-216: fp32 features [B,N,Dc], int64 tokens [B,N,1], int64 mask [B,N,1]; result on the host).
 * The jets are cut into n_chunks slices that travel through internal streams: H2D of slice c+1 and D2H of slice c-1 run under
 * the solver steps of slice c; tokens / masks are narrowed to uint8 and widened back on the device; Philox is keyed by the
 * global jet index, so the result equals the unsliced call bit for bit.
 *   x_in, k_in, mask_in, context_in (nullable, [B,X]), x_out, k_out, bad_tokens: HOST pointers (page-locked for the copies to
 *   be asynchronous; x_out / k_out may alias x_in / k_in).  *bad_tokens becomes 1 if any input token lies outside [0, S) — the reference asserts that
 *   (bridges.py:111-115); the caller raises after synchronising.  In-kernel Philox only.
 *   n_chunks <= 0 selects the DIRECT mode (MMB_PREC_F16 with page-locked buffers; anything else falls back to two slices):
 *   no slicing and no staging copies of features or tokens — each warp of the generation kernel reads the source state of the
 *   jet it claims straight from the mapped host buffers and writes the final state straight back, so the PCIe traffic of a
 *   jet hides under the solver steps of the others; only the masks (needed up front to order the jets) and a copy of the
 *   tokens for the range assertion travel by DMA, on side streams.
 *   workspace: mmb_generate_host_workspace_bytes(...) bytes of 256-byte aligned DEVICE memory.
 * Asynchronous: everything is ordered after the work already on `stream`, and `stream` continues after the last copy;
 * results are valid once the caller has synchronised `stream`.  Streams and events are created on the first call.
 */
size_t mmb_generate_host_workspace_bytes(const MmbEpicModel* m, int B, int N, int n_steps, int n_chunks, int precision);
int mmb_generate_host(const MmbEpicModel* m, const float* x_in, const int64_t* k_in, const int64_t* mask_in,
                      const float* context_in, const MmbStepTable* st, uint64_t seed, uint64_t jet_offset, int B, int N,
                      float* x_out, int64_t* k_out, int32_t* bad_tokens, void* workspace, size_t workspace_bytes,
                      int n_chunks, int precision, void* stream);

/*
 * Diagnostics: the jump rule (TelegraphBridge.solver_step, bridges.py:179-201, as the one-uniform categorical) evaluated by
 * its three device implementations on IDENTICAL inputs — the exact rule of MMB_PREC_FP32 / mmb_bridge_update (bit-identical to
 * the oracle) and the fast-intrinsic variants inside the MMB_PREC_BF16 and MMB_PREC_F16 generation kernels.
 *   logits [P,S] f32, k [P] u8, u [P] f32 -> new tokens out_exact / out_tc / out_mma [P] u8 (unmasked).  S in {4, 8}.
 */
int mmb_jump_variants(const float* logits, const uint8_t* k, const float* u, float dt, float bc, float cc, size_t P, int S,
                      uint8_t* out_exact, uint8_t* out_tc, uint8_t* out_mma, void* stream);

/* uniforms exactly as the in-kernel generator draws them, written to u [n_steps,B,N] (for tests) */
int mmb_philox_uniforms(float* u, uint64_t seed, uint64_t jet_offset, int n_steps, int B, int N, void* stream);

/*
 * Absorbing-rate transformer head of AbsorbingGenerator (mp/models/generative/absorbing/absorbing_flows.py:56-131;
 * blocks: mp/models/architectures/gsdm.py:38-66,142-168).  Built for transformer_dim = 128, n_heads = 2.
 * Packed blob (fp32, every matrix row-major [out][in] followed by its bias):
 *   transformer_1_proj_in [C][H+2]+[C];
 *   per block: res.norm1 g[C] b[C]; res.conv1 [C][C]+[C]; res.norm2 g b; res.conv2 [C][C]+[C];
 *              attn.norm g b; attn.q [C][C]+[C]; attn.k; attn.v; attn.proj_out;
 *   pre_rate_proj [C][C]+[C]; post_rate_proj [1][C]+[1].
 * The time term of every ResnetBlock, temb_proj_b(swish(temb_net(timestep_embedding(1000 t)))), is an input
 * (tbias [B or 1][n_blocks][C], stride 0 = one time for all jets): at generation time it is a per-step constant
 * the host computes once per step table.
 */
typedef struct MmbAbsorbHead MmbAbsorbHead;
int mmb_absorb_head_create(int hidden, int transformer_dim, int n_heads, int n_blocks, const float* packed, size_t n_floats,
                           int device, MmbAbsorbHead** out);
void mmb_absorb_head_destroy(MmbAbsorbHead* head);
/*
 * hidden [B,N,H] (EPiC last local hidden), mask [B,N] u8 -> logit_out [B,N] (heads.absorbing[...,0]).
 * The reference runs the stack over all N slots, padded ones included (no attention mask, GroupNorm over every slot).  With a
 * workspace of mmb_absorb_head_workspace_bytes(B) bytes (device, 4-byte aligned) the kernel computes the identical padded
 * slots of a jet ONCE (a representative row carrying the weight n_dead in every sum over slots — exact) and packs several jets
 * into one 128-row tile with block-diagonal attention; jets whose padded slots do not hold identical inputs keep one row per
 * slot.  workspace = NULL: one jet per tile, one row per slot.
 */
size_t mmb_absorb_head_workspace_bytes(int B);
int mmb_absorb_head_forward(const MmbAbsorbHead* head, const float* hidden, const uint8_t* mask, const float* tbias,
                            int tbias_stride, int B, int N, float* logit_out, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Whole generation loop of the absorbing flow: per step trunk + discrete head (mmb_epic_forward with the last
 * hidden), rate head, then mmb_bridge_update(MMB_FLAG_ABSORBING).  Stands behind AbsorbingFlow.simulate_dynamics
 * (absorbing_flows.py:255-275) minus the final .cpu().  mask is in/out (particles are born).
 *   tbias: HOST [n_steps][n_blocks][C];  u_jump / u_absorb: device [n_steps,B,N] or NULL for Philox streams 0 / 1.
 */
size_t mmb_generate_absorbing_workspace_bytes(const MmbEpicModel* model, const MmbAbsorbHead* head, int B, int N, int n_steps);
int mmb_generate_absorbing(const MmbEpicModel* model, const MmbAbsorbHead* head, float* x, uint8_t* k, uint8_t* mask,
                           const MmbStepTable* steps, const float* tbias, const float* u_jump, const float* u_absorb,
                           uint64_t seed, uint64_t jet_offset, int B, int N, void* workspace, size_t workspace_bytes,
                           int precision, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Trans-dimensional jump diffusion (BASELINE config "transepic"; SURVEY.md §8a rows A12, A13).
 *
 * TransdimensionalEPiC.forward (mp/models/generative/transdimensional/transdimensional_model.py:245-426,
 * called through EpsilonPrecond.forward :124-133): EPiC trunk with the last local hidden, then two
 * 128-wide transformer stacks (gsdm.py ResnetBlock + AttnBlock): the first gives the per-jet x0-dimension
 * logits (hence the birth rate, mp/models/generative/diffusion/noising.py:166-216) and the nearest-particle
 * logits, the second — fed with the distance to the chosen nearest particle — gives mean and std of the
 * particle that a birth adds.
 */
typedef struct MmbTransDims {
    int32_t hidden;          /* H  encoder.dim_hidden_local (width of the trunk's last local hidden) */
    int32_t vocab_size;      /* S  data.vocab_size_features (one-hot channels) */
    int32_t transformer_dim; /* C  encoder.transformer_dim (= temb_dim); built for 128 */
    int32_t n_heads;         /*    encoder.n_heads; built for 2 */
    int32_t n_blocks;        /*    encoder.n_attn_blocks */
    int32_t max_particles;   /* R  data.max_num_particles: width of x0_dim_logits, rdim of post_rate_proj when rate_direct == 0 */
    int32_t rate_direct;     /* 1: encoder.rate_use_x0_pred = False — post_rate_proj has ONE output, rate = softplus(.) * forward_rate(t)
                                and x0_dim_logits = 0 (transdimensional_model.py:185-188, 326-332); 0: every shipped config */
} MmbTransDims;

/* StepForwardRate / ConstForwardRate (noising.py:123-164): rate(t) = scalar*[t > cut] + offset (step),
 * scalar (const);  integral(t) = (t-cut)*scalar*[t > cut] + offset*t (step), scalar*t (const). */
typedef struct MmbForwardRate {
    int32_t kind;  /* 0 = step, 1 = const */
    float scalar, offset, rate_cut_t;
} MmbForwardRate;

/*
 * Packed blob (fp32, every matrix row-major [out][in] followed by its bias), C = transformer_dim:
 *   temb_net [C][C]+[C];
 *   res_blocks[i].temb_proj [C][C]+[C], i < n_blocks;  vec_res_blocks[i].temb_proj [C][C]+[C], i < n_blocks;
 *   stack 1: transformer_1_proj_in [C][H+S]+[C]; n_blocks x block; pre_rate_proj [C][C]+[C];
 *            post_rate_proj [R][C]+[R]; near_atom_proj [1][C]+[1];
 *   stack 2: vec_transformer_in_proj [C][H+S+3]+[C]; n_blocks x block; vec_weighting_proj [1][C]+[1];
 *            pre_auto_proj [C][C]+[C]; post_auto_proj [2S+1][C]+[2S+1];
 * with block = res.norm1 g b; res.conv1; res.norm2 g b; res.conv2; attn.norm g b; attn.q; attn.k; attn.v; attn.proj_out
 * (the block layout of mmb_absorb_head_create).
 */
typedef struct MmbTransHeads MmbTransHeads;
size_t mmb_trans_packed_floats(const MmbTransDims* dims);
int mmb_trans_create(const MmbTransDims* dims, const float* packed, size_t n_floats, int device, MmbTransHeads** out);
void mmb_trans_destroy(MmbTransHeads* heads);

/*
 * One network evaluation = EpsilonPrecond.forward(st_batch, ts, predict='eps', forward_rate, nearest_atom)
 * (transdimensional_model.py:124-133 -> :245-426), including StructuredDataBatch.
 * from_st_batch_to_multimodal_bridge_databatch (structure.py:226-250: tokens = argmax of the one-hot block after
 * F.softmax WITHOUT dim, i.e. over the BATCH axis of the 3-D tensor; prefix mask from dims).
 *   x [B,N,3], onehot [B,N,S] (the latent tuple_batch), dims [B] int32 (1..N), ts [B];
 *   nearest_in [B] int32, or NULL to sample it from softmax(near_atom_logits) over all N slots with the
 *   uniform u_nearest [B] (inverse CDF; replaces rnd.multinomial, transdimensional_model.py:335-339);
 *   trunk: an MmbEpicModel created with disc_head_hidden = 0 (fc_layer is constructed but never applied).
 * Outputs: d_xt [B, N*(3+S)] (all continuous slots, then all one-hot slots, :277-280), rate [B],
 *   auto_mean / auto_std [B, N*(3+S)] (zero outside slot `dims`; NULL = skip), x0_dim_logits [B,R],
 *   near_atom_logits [B,N], nearest_out [B] int32 (NULL = skip).
 */
size_t mmb_trans_forward_workspace_bytes(const MmbEpicModel* trunk, const MmbTransHeads* heads, int B, int N);
int mmb_trans_forward(const MmbEpicModel* trunk, const MmbTransHeads* heads,
                      const float* x, const float* onehot, const int32_t* dims, const float* ts,
                      const int32_t* nearest_in, const float* u_nearest, const MmbForwardRate* forward_rate,
                      int B, int N,
                      float* d_xt, float* rate, float* auto_mean, float* auto_std, float* x0_dim_logits,
                      float* near_atom_logits, int32_t* nearest_out,
                      void* workspace, size_t workspace_bytes, int precision, void* stream);

/*
 * JumpSampler.sample (mp/models/generative/transdimensional/sampler.py:157-324; sample_near_atom, no conditioning) —
 * reverse VP-SDE Euler-Maruyama on the flat latents with a birth jump per step, optionally followed by Langevin
 * corrector evaluations (sampler.py:258-282) with their own birth/death jumps (do_jump_corrector, :285-312).
 * The schedule is a host table with one ROW PER NETWORK EVALUATION, computed with torch fp32 ops in the reference's
 * order (all jets share ts):
 *   predictor row (kind 0): ts, c_decay = 2 - sqrt(1 - beta dt), c_score = beta dt, c_noise = sqrt(beta dt) (0 where
 *     the reference adds no noise: no_noise_final_step), inv_std = 1/clamp(std(ts), 1e-3);
 *   corrector row (kind 1): ts = t - dt, c_score = alpha = 1 - dt beta(t - dt), c_noise = 1 (0: the final corrector
 *     under no_noise_final_step), inv_std at t - dt, death_prob = forward_rate(t - dt) dt; c_decay unused.  The step
 *     size (corrector_snr * mean_b|noise_b| / mean_b|score_b|)^2 * 2 alpha is a batch statistic computed on the device.
 * jump_dt = dt.  kind == NULL means predictor rows only.
 * State in/out: x [B,N,3], onehot [B,N,S], dims [B] int32 — the caller initialises them like sampler.py:170-183
 * (x_T ~ N(0,I), dims = 1, delete_dims, adjust_st_batch) or passes any intermediate state.
 * Noise: either injected (device pointers indexed by row; parity runs)
 *   z_diff [n_steps][B][N*(3+S)] (rnd.randn_like(xt)), u_near [n_steps][B], u_jump [n_steps][B],
 *   z_new [n_steps][B][3+S] (the draw that lands in the new slot), u_death [n_steps][B] (jump corrector only, else NULL),
 * or all NULL: in-kernel Philox4x32-10 keyed by (seed, jet_offset + jet, row, element) + Box-Muller.
 */
typedef struct MmbJumpSchedule {
    int32_t n_steps;       /* rows = network evaluations */
    const float* ts;       /* HOST [n_steps] */
    const float* c_decay;  /* HOST [n_steps] */
    const float* c_score;  /* HOST [n_steps] */
    const float* c_noise;  /* HOST [n_steps] */
    const float* inv_std;  /* HOST [n_steps] */
    float jump_dt;
    const uint8_t* kind;     /* HOST [n_steps] or NULL */
    const float* death_prob; /* HOST [n_steps] or NULL (needed when jump_corrector) */
    float corrector_snr;
    int32_t jump_corrector;
} MmbJumpSchedule;
size_t mmb_trans_sample_workspace_bytes(const MmbEpicModel* trunk, const MmbTransHeads* heads, int B, int N);
int mmb_trans_sample(const MmbEpicModel* trunk, const MmbTransHeads* heads, float* x, float* onehot, int32_t* dims,
                     const MmbJumpSchedule* schedule, const MmbForwardRate* forward_rate,
                     const float* z_diff, const float* u_near, const float* u_jump, const float* z_new, const float* u_death,
                     uint64_t seed, uint64_t jet_offset, int B, int N,
                     void* workspace, size_t workspace_bytes, int precision, void* stream);
/* one sampler update alone (sampler.py:221-255 + adjust_st_batch, jets_dataloader.py:433-478): the fused,
 * HBM-bound kernel of the loop.  v [B,N,3], logits [B,N,S] are the two halves of D_xt; new_mean/new_std [B][3+S]
 * the compact mean/std of the slot a birth fills; step selects the Philox counters when the noise pointers are NULL. */
int mmb_trans_sampler_update(float* x, float* onehot, int32_t* dims, const float* v, const float* logits, const float* rate,
                             const float* new_mean, const float* new_std,
                             float c_decay, float c_score, float c_noise, float inv_std, float jump_dt,
                             const float* z_diff, const float* u_jump, const float* z_new,
                             uint64_t seed, uint64_t jet_offset, int step, int B, int N, int S, void* stream);
/* one Langevin corrector update alone (sampler.py:258-282; with jump_corrector also :285-312): batch norms of the
 * score and of the centred noise -> step size -> increment on the slots the predictor step's mask covers
 * (mask_dims [B], NULL = dims) -> centre-of-mass removal -> optional birth/death.  alpha = 1 - dt beta(t - dt);
 * scratch: 2B + 4 device floats (scratch[2B+3] returns the step size). */
int mmb_trans_corrector_update(float* x, float* onehot, int32_t* dims, const int32_t* mask_dims, const float* v, const float* logits,
                               const float* rate, const float* new_mean, const float* new_std, float alpha, int noise_on, float inv_std,
                               float corrector_snr, float jump_dt, int jump_corrector, float death_prob, const float* z_diff,
                               const float* u_jump, const float* u_death, const float* z_new, uint64_t seed, uint64_t jet_offset, int step,
                               int B, int N, int S, float* scratch, void* stream);

/*
 * Validation histograms of a generated batch, ACCUMULATED into counts (caller zeroes it): the
 * per-GPU buffer that the multi-GPU layer all-reduces (SURVEY.md §8e).  Layout of counts (uint64):
 *   [Dc][bins] per-particle histograms of the continuous features over [lo,hi) (out-of-range values
 *   go to the edge bins) | [S] token counts | [max_mult+1] particle multiplicity per jet (clamped).
 * Only live particles (mask != 0) are counted.  Stands behind the jet-level observables of
 * JetClassHighLevelFeatures that need no clustering (mp/data/particle_clouds/jets.py:90-107).
 */
int mmb_validation_histograms(const float* x, const uint8_t* k, const uint8_t* mask, int B, int N, int Dc, int S,
                              int bins, float lo, float hi, int max_mult, uint64_t* counts, void* stream);

/*
 * Post-processing + jet-level observables of a generated batch in one pass (SURVEY.md §8f N1), so that validation needs the
 * 44-byte jet rows instead of the particle clouds:
 *   ParticleClouds.postprocess(input_continuous="standardize", input_discrete="tokens")  (mp/data/particle_clouds/particles.py:124-156):
 *     x_phys = (x * std + mean) * mask;  tokens_to_physics (mp/data/particle_clouds/utils.py:310-337): flavor 0..4, charge -1/0/+1, both * mask;
 *   ParticleClouds.compute_4mom (particles.py:85-89) and JetClassHighLevelFeatures.__init__ / jet_charge
 *     (mp/data/particle_clouds/jets.py:90-107,138-141): per jet px, py, pz, e (sums over ALL slots of the masked cloud),
 *     pt = sqrt(max(px^2+py^2, 0)), m = sqrt(max(e^2-px^2-py^2-pz^2, 0)), eta = 0.5 log((pt+pz)/(pt-pz)), phi = atan2(py, px),
 *     multiplicity, Q_total = sum charge, Q_jet = sum charge*pt / pt_jet.
 * x [B,N,3] f32, k [B,N] u8 tokens (0..7), mask [B,N] u8; mean / std: HOST float[3], or NULL for data that is not standardised.
 * Outputs (each nullable): x_phys [B,N,3] f32; flavor_charge [B,N,2] int8 (flavor, charge; 0,0 on masked slots);
 * jets [B][MMB_JET_OBS] f32 in the order of the enum below.
 */
enum { MMB_JET_PX = 0, MMB_JET_PY, MMB_JET_PZ, MMB_JET_E, MMB_JET_PT, MMB_JET_M, MMB_JET_ETA, MMB_JET_PHI, MMB_JET_MULT,
       MMB_JET_QTOTAL, MMB_JET_QJET, MMB_JET_OBS };
int mmb_jet_observables(const float* x, const uint8_t* k, const uint8_t* mask, const float* mean, const float* std, int B, int N,
                        float* x_phys, int8_t* flavor_charge, float* jets, void* stream);

/*
 * Jet substructure of a generated batch (the clustering-based observables of JetClassHighLevelFeatures.substructure,
 * mp/data/particle_clouds/jets.py:204-240), so that validation on tau21, tau32 and D2 needs the 32-byte rows, not the clouds:
 *   constituents (pt, eta, phi) = (x * std + mean) in fp32 (mean / std: HOST float[3], or NULL for physical input), massless;
 *   a particle is used iff mask != 0 && pt > 0.
 *   Exclusive kt clustering with WTA_pt recombination over the used particles, in fp64 without contraction:
 *     d_ij = min(pt_i^2, pt_j^2) dR_ij^2 (1 / R^2) (dphi wrapped into [-pi, pi]), d_iB = pt_i^2; each step takes the minimum of
 *     all d_ij and d_iB, ties to the smaller (lower, upper) index pair, a beam candidate being (i, i).  A pair merges into the
 *     lower index with pt_i + pt_j and the direction of the harder one (lower index on a pt tie); a beam step removes the
 *     object.  The exclusive n-jet axes are the objects left when n remain (n = 3, 2, 1).
 *   tau_N = sum_i pt_i min_a dR(i,a)^beta / sum_i pt_i R^beta;  tau21 = tau2 / tau1, tau32 = tau3 / tau2;
 *   with z_i = pt_i / sum_j pt_j (arXiv:1409.6298): e2 = sum_{i<j} z_i z_j dR_ij^beta,
 *   e3 = sum_{i<j<k} z_i z_j z_k (dR_ij dR_ik dR_jk)^beta, D2 = e3 / e2^3.
 * A jet with fewer than 3 used particles gets NaN in every column and axes -1; 0/0 ratios are NaN.
 * x [B,N,3] f32, mask [B,N] u8, N <= 256 (larger N: MMB_EINVAL); R > 0, beta > 0.
 * Outputs: out [B][MMB_SUB_OBS] f32 in the order of the enum below; axes [B][6] int16 (nullable): the particle slot (0..N-1)
 * whose direction is each WTA axis — tau1 axis | tau2 axes | tau3 axes, each set in ascending order of its object's slot.
 */
enum { MMB_SUB_TAU1 = 0, MMB_SUB_TAU2, MMB_SUB_TAU3, MMB_SUB_TAU21, MMB_SUB_TAU32, MMB_SUB_E2, MMB_SUB_E3, MMB_SUB_D2, MMB_SUB_OBS };
#define MMB_SUB_MAX_N 256
int mmb_jet_substructure(const float* x, const uint8_t* mask, const float* mean, const float* std, int B, int N, float R, float beta,
                         float* out, int16_t* axes, void* stream);

/*
 * 1-D Wasserstein distance per column between two samples (JetClassHighLevelFeatures.Wassertein1D, jets.py:329-332, which is
 * scipy.stats.wasserstein_distance), so that scoring generated jets against a reference needs no host copy of either sample:
 *   the non-finite values (NaN, +-inf) of each column are dropped and counted out; n' and m' finite x and y values remain;
 *   z_0 <= z_1 <= ... is the merged sorted sequence of both, i_k and j_k the numbers of x and y values <= z_k;
 *   W1 = sum_k |i_k m' - j_k n'| (z_{k+1} - z_k) / (n' m'),  |i_k m' - j_k n'| exact in int64, differences and sum in fp64;
 *   n' = 0 or m' = 0: NaN.
 * Radix sort of each column (CUB), merge-path integration in fixed tiles, fixed-order sums: the result is bit-identical from
 * call to call and for any order of the rows.
 * x: row r, column c at x[r*ldx + c] (ldx >= K), n rows; y likewise with ldy, m rows; device f32 (NULL allowed for 0 rows).
 * out [K] f64 (device): W1 per column over the finite values; n_used [2K] int64 (device, nullable): finite x values per column,
 * then finite y values per column.  0 < K <= MMB_W1_MAX_K, 0 <= n, m <= 2^31 - 1, else MMB_EINVAL.  workspace: 256-byte aligned,
 * mmb_wasserstein1d_workspace_bytes(n, m, K) bytes (0 for invalid sizes), else MMB_ENOMEM.
 */
#define MMB_W1_MAX_K 64
size_t mmb_wasserstein1d_workspace_bytes(int n, int m, int K);
int mmb_wasserstein1d(const float* x, int64_t ldx, int n, const float* y, int64_t ldy, int m, int K,
                      double* out, int64_t* n_used, void* workspace, size_t workspace_bytes, void* stream);

/*
 * The same W1 per draw and feature over the used slots of drawn jets (JetNet's W1-P, and with P = 1 and no masks its W1-M and
 * W1-EFP draws, arXiv:2211.10295), with no host copy of the drawn samples and no host synchronisation:
 *   value of jet j, slot p, feature c: x[j*ldx_jet + p*ldx_slot + c]; the slot is used iff mask_x == NULL || mask_x[j*ldmx + p];
 *   the sample of draw t is the used slots of the jets idx_x[t][0..rows), in draw order and within a jet in slot order (a jet
 *   drawn k times contributes k times); y, mask_y, idx_y likewise;
 *   out [draws][F] f64 (device): out[t][c] is bit-identical to mmb_wasserstein1d on the two samples of draw t gathered into
 *   rows (non-finite values dropped, NaN when a sample has no finite value); n_used [2][draws][F] int64 (device, nullable):
 *   finite x values, then finite y values.
 * 0 < F <= MMB_W1_MAX_K, P >= 1, draws >= 1, rows >= 1, rows * P <= 2^31 - 1, 2 * draws * F <= 2^31 - 1, n, m >= 1, ldx_slot >= F (P > 1),
 * ldx_jet >= (P - 1) * ldx_slot + F, ldmx >= P with a mask (y likewise), else MMB_EINVAL.  Jet indices are device int32
 * [draws][rows] in [0, n) / [0, m) (not checked).  workspace: 256-byte aligned, mmb_wasserstein1d_drawn_workspace_bytes(draws,
 * rows, P, F) bytes (0 for invalid sizes), else MMB_ENOMEM.  Stream-ordered, allocates nothing, bit-identical from call to call.
 */
size_t mmb_wasserstein1d_drawn_workspace_bytes(int draws, int rows, int P, int F);
int mmb_wasserstein1d_drawn(const float* x, int64_t ldx_jet, int64_t ldx_slot, const uint8_t* mask_x, int64_t ldmx, int n,
                            const float* y, int64_t ldy_jet, int64_t ldy_slot, const uint8_t* mask_y, int64_t ldmy, int m,
                            int P, int F, const int32_t* idx_x, const int32_t* idx_y, int draws, int rows,
                            double* out, int64_t* n_used, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Energy flow polynomials of a generated batch (the features of the W1-EFP, FPD and KPD metrics, arXiv:2211.10295, as JetNet
 * computes them with energyflow: hadronic measure, kappa = 1, normalised energies):
 *   constituents as for mmb_jet_substructure ((x * std + mean) in fp32, massless, y = eta; used iff mask != 0 && pt > 0);
 *   z_i = pt_i / sum_j pt_j over the used particles, theta_ij = dR_ij^beta (dphi wrapped into [-pi, pi]), theta_ii = 0;
 *   EFP_G = sum over all index tuples (coincident indices included) of z_i1 ... z_iV prod_{(a,b) in G} theta_{ia ib}.
 * With s_i = sum_j z_j theta_ij, q_i = sum_j z_j theta_ij^2 and M = Theta diag(z) Theta, the columns are
 *   EFP_1            one edge                          sum_i z_i s_i
 *   EFP_4_SQUARE     4-cycle                           sum_{i,k} z_i z_k M_ik^2
 *   EFP_4_PAW        triangle plus pendant             sum_i z_i s_i sum_k z_k theta_ik M_ik
 *   EFP_4_PATH_MID2  3-edge path, middle edge doubled  sum_{j,k} z_j z_k s_j theta_jk^2 s_k
 *   EFP_4_PATH_END2  3-edge path, end edge doubled     sum_{j,k} z_j z_k q_j theta_jk s_k
 *   EFP_4_STAR2      3-star, one edge doubled          sum_i z_i q_i s_i^2
 * (the last five are every connected multigraph with 4 vertices and 4 edges).  theta and M are fp32, every sum fp64.
 * A jet with no used particle gets NaN in every column (one used particle: 0).
 * x [B,N,3] f32, mask [B,N] u8, N <= MMB_SUB_MAX_N (larger N: MMB_EINVAL); beta > 0.  out [B][MMB_EFP_OBS] f32.
 * Bit-identical from call to call.
 */
enum { MMB_EFP_1 = 0, MMB_EFP_4_SQUARE, MMB_EFP_4_PAW, MMB_EFP_4_PATH_MID2, MMB_EFP_4_PATH_END2, MMB_EFP_4_STAR2, MMB_EFP_OBS };
int mmb_energy_flow_polynomials(const float* x, const uint8_t* mask, const float* mean, const float* std, int B, int N, float beta,
                                float* out, void* stream);

/*
 * Every energy flow polynomial of degree (edge count) d <= 4: the feature set JetNet scores FPD and KPD on (efpset ("d<=", 4),
 * 36 EFPs).  Constituents, z, theta and the index-tuple sum as for mmb_energy_flow_polynomials; in addition
 *   c_i = sum_j z_j theta_ij^3, r_i = sum_j z_j theta_ij^4, u_i = sum_k theta_ik z_k s_k.
 * The 20 connected loopless multigraphs with 1 <= d <= 4 (V vertices):
 *   d = 1  EFPD4_1                  edge (V 2)                       sum_i z_i s_i
 *   d = 2  EFPD4_2_DOUBLE           double edge (2)                  sum_i z_i q_i
 *          EFPD4_2_PATH             2-edge path (3)                  sum_i z_i s_i^2
 *   d = 3  EFPD4_3_TRIPLE           triple edge (2)                  sum_i z_i c_i
 *          EFPD4_3_PATH_DOUBLE      2-edge path, one edge doubled (3) sum_i z_i q_i s_i
 *          EFPD4_3_TRIANGLE         triangle (3)                     sum_{i,k} z_i z_k theta_ik M_ik
 *          EFPD4_3_PATH             3-edge path (4)                  sum_i z_i s_i u_i
 *          EFPD4_3_STAR             3-star (4)                       sum_i z_i s_i^3
 *   d = 4  EFPD4_4_QUADRUPLE        quadruple edge (2)               sum_i z_i r_i
 *          EFPD4_4_TRIPLE_SINGLE    triple edge + edge (3)           sum_i z_i c_i s_i
 *          EFPD4_4_DOUBLE_DOUBLE    two doubled edges (3)            sum_i z_i q_i^2
 *          EFPD4_4_TRIANGLE_DOUBLE  triangle, one edge doubled (3)   sum_{i,k} z_i z_k theta_ik^2 M_ik
 *          EFPD4_4_SQUARE .. EFPD4_4_STAR2   the five 4-vertex graphs of mmb_energy_flow_polynomials, same formulas
 *          EFPD4_4_PATH             4-edge path (5)                  sum_i z_i u_i^2
 *          EFPD4_4_STAR             4-star (5)                       sum_i z_i s_i^4
 *          EFPD4_4_FORK             3-star, one leg extended (5)     sum_i z_i s_i^2 u_i
 * and the empty graph EFPD4_0 = 1 and the 15 disconnected graphs, whose EFP is the product of their components' (formed in
 * fp64 from the fp64 sums, rounded once): EFPD4_1_1 is efp1^2, EFPD4_1_2_DOUBLE is efp1 * efp2_double, and so on; the
 * columns are ordered by d, connected before disconnected.  EFPD4_1 and the five EFPD4_4_{SQUARE, PAW, PATH_MID2, PATH_END2,
 * STAR2} are bit-identical to the columns of mmb_energy_flow_polynomials on the same input and beta.
 * A jet with no used particle gets NaN in every column; one used particle: EFPD4_0 = 1, every other column 0.
 * x [B,N,3] f32, mask [B,N] u8, N <= MMB_SUB_MAX_N (larger N: MMB_EINVAL); beta > 0.  out [B][MMB_EFPD4_OBS] f32.
 * Stream-ordered, allocates nothing, bit-identical from call to call.
 */
enum {
    MMB_EFPD4_0 = 0,
    MMB_EFPD4_1,
    MMB_EFPD4_2_DOUBLE, MMB_EFPD4_2_PATH, MMB_EFPD4_1_1,
    MMB_EFPD4_3_TRIPLE, MMB_EFPD4_3_PATH_DOUBLE, MMB_EFPD4_3_TRIANGLE, MMB_EFPD4_3_PATH, MMB_EFPD4_3_STAR,
    MMB_EFPD4_1_2_DOUBLE, MMB_EFPD4_1_2_PATH, MMB_EFPD4_1_1_1,
    MMB_EFPD4_4_QUADRUPLE, MMB_EFPD4_4_TRIPLE_SINGLE, MMB_EFPD4_4_DOUBLE_DOUBLE, MMB_EFPD4_4_TRIANGLE_DOUBLE, MMB_EFPD4_4_SQUARE,
    MMB_EFPD4_4_PAW, MMB_EFPD4_4_PATH_MID2, MMB_EFPD4_4_PATH_END2, MMB_EFPD4_4_STAR2, MMB_EFPD4_4_PATH, MMB_EFPD4_4_STAR,
    MMB_EFPD4_4_FORK,
    MMB_EFPD4_1_3_TRIPLE, MMB_EFPD4_1_3_PATH_DOUBLE, MMB_EFPD4_1_3_TRIANGLE, MMB_EFPD4_1_3_PATH, MMB_EFPD4_1_3_STAR,
    MMB_EFPD4_2_DOUBLE_2_DOUBLE, MMB_EFPD4_2_DOUBLE_2_PATH, MMB_EFPD4_2_PATH_2_PATH, MMB_EFPD4_1_1_2_DOUBLE, MMB_EFPD4_1_1_2_PATH,
    MMB_EFPD4_1_1_1_1,
    MMB_EFPD4_OBS
};
int mmb_energy_flow_polynomials_d4(const float* x, const uint8_t* mask, const float* mean, const float* std, int B, int N,
                                   float beta, float* out, void* stream);

/*
 * Sample statistics of the Frechet and kernel physics distances (FPD, KPD; arXiv:2211.10295) over rows the caller draws:
 * x: row r, column c at x[r*ldx + c] (ldx >= d), n rows, device f32; every value is used as x * scale[c] in fp64 (scale: device
 * f32 [d], NULL for 1).  Row indices are device int32 in [0, n) (not checked).  0 < d <= MMB_MET_MAX_D.
 *
 * mmb_sampled_moments: for each draw t, over the rows idx[t][0..rows): sum[t][a] = sum x_a, sumsq[t][a][b] = sum x_a x_b
 * (both triangles written), fp64 on the device.  draws > 0, rows > 0.
 *
 * mmb_kpd_mmd: for each batch t, with r_i = real[idx_real[t][i]], g_j = gen[idx_gen[t][j]] (i, j < B) and
 * k(u, v) = (u . v / d + 1)^degree, the unbiased MMD^2
 *   out[t] = (sum_{i != j} k(r_i, r_j) + sum_{i != j} k(g_i, g_j)) / (B (B - 1)) - 2 sum_{i,j} k(r_i, g_j) / B^2,
 * dot products, powers and sums in fp64.  batches in 1..65535, B >= 2, degree >= 1.  workspace: 256-byte aligned,
 * mmb_kpd_mmd_workspace_bytes(batches, B, d) bytes (0 for invalid sizes), else MMB_ENOMEM.
 * Both are stream-ordered, allocate nothing and are bit-identical from call to call.
 */
#define MMB_MET_MAX_D 64
int mmb_sampled_moments(const float* x, int64_t ldx, int n, int d, const float* scale, const int32_t* idx, int draws, int rows,
                        double* sum, double* sumsq, void* stream);
size_t mmb_kpd_mmd_workspace_bytes(int batches, int B, int d);
int mmb_kpd_mmd(const float* real, int64_t ldr, int n, const float* gen, int64_t ldg, int m, int d, const float* scale,
                const int32_t* idx_real, const int32_t* idx_gen, int batches, int B, int degree, double* out, void* workspace,
                size_t workspace_bytes, void* stream);

/*
 * Source-state construction on the device (SURVEY.md §8f N3), so that a generation run needs no host data loader:
 *   sample_noise("GaussNoise") (mp/data/particle_clouds/utils.py:222-251): x ~ N(0,1) * scale, flavor ~ Categorical(cat_probs[5]),
 *   charge = +-1 (0 for photons / neutral hadrons), turned into the 8 tokens of physics_to_onehot + argmax
 *   (utils.py:289-307; ParticleClouds.preprocess "tokens", particles.py:111-113);
 *   sample_masks (utils.py:254-286): multiplicity ~ Categorical(histogram of the target multiplicities), prefix mask;
 *   x and k are multiplied by the mask (particles.py:65-69).
 * Draws come from Philox4x32-10 keyed by (seed, jet_offset + jet, particle) — streams 9 (normals) and 10 (flavor, charge),
 * 11 (multiplicity) — so a sharded run produces the same jets as a single-GPU run.
 *   cat_probs: HOST float[5];  mult_cdf: DEVICE float[N+1] cumulative multiplicity probabilities (m = first i with u < cdf[i]),
 *   or NULL for full jets.  Outputs: x [B,N,3] f32, k [B,N] u8, mask [B,N] u8.
 */
int mmb_sample_source(float* x, uint8_t* k, uint8_t* mask, int B, int N, float scale, const float* cat_probs, const float* mult_cdf,
                      uint64_t seed, uint64_t jet_offset, void* stream);

/*
 * Forward half of a training / validation step (SURVEY.md §8f N2) — bridge sampling and the masked losses; the backward pass
 * stays out of scope.
 *
 * mmb_sample_bridges = MultiModalBridgeMatching.sample_bridges (mp/models/generative/multimodal_bridge_matching.py:148-165) given the
 * per-jet times t [B]:  xt = (t x1 + (1-t) x0) + sigma z  (LinearUniformBridge.sample, bridges.py:23-27);
 * kt ~ Categorical(P(k | k0, k1, t)) with the telegraph-bridge posterior (TelegraphBridge.sample, bridges.py:99-104,134-177),
 * drawn by inverse CDF on one uniform per particle.  z [B,N,3] / u [B,N] inject the draws (both or neither); NULL = Philox
 * streams 12/13 keyed by (seed, jet_offset + jet, particle).
 */
int mmb_sample_bridges(const float* x0, const float* x1, const uint8_t* k0, const uint8_t* k1, const float* t, float sigma, float gamma,
                       int S, const float* z, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N,
                       float* xt, uint8_t* kt, void* stream);
/* AbsorbingBridge.sample (bridges.py:233-249): mask_t = [u < SP(t)] | target_mask, sp [B] = survival probability at each jet's time
 * (bridges.py:218-231, computed by the caller); u [B,N] or NULL for Philox stream 14. */
int mmb_absorbing_sample(const float* sp, const uint8_t* target_mask, const float* u, uint64_t seed, uint64_t jet_offset, int B, int N,
                         uint8_t* mask_t, void* stream);
/*
 * loss_continuous + loss_discrete (multimodal_bridge_matching.py:167-197): masked MSE between the velocity head and the drift
 * target x1 - x0, masked cross entropy between the logits and the target tokens, both divided by the number of live particles.
 * out [3] (device) = { mse, ce, live particles }.  workspace: mmb_bridge_losses_workspace_bytes(B, N) bytes.
 * Sums are reduced in a fixed order (deterministic).
 */
size_t mmb_bridge_losses_workspace_bytes(int B, int N);
int mmb_bridge_losses(const float* v, const float* logits, const float* x0, const float* x1, const uint8_t* k1, const uint8_t* mask,
                      int B, int N, int S, float* out, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMBRIDGE_H */
