// epic_grad.cu — the bridge-matching losses of MultiModalBridgeMatching and their gradients with respect to every weight of
// the packed EPiC blob, fp32 on CUDA cores (mbm.py:167-197, 232-240; epic.py:136-241; utils.py:112-172).
//
// epic_loss_grad_kernel: a persistent grid of P CTAs of 128 threads; CTA c takes jets c, c+P, ... in ascending order.  Per jet
// it recomputes the forward in the IEEE operation order of epic_forward_jet (epic_fp32.cu), so its heads are those of
// mmb_epic_forward(precision = fp32), keeps every activation the backward needs in the CTA's region of the workspace, forms
// the per-particle loss terms, and runs the backward twice: once seeded with the MSE head gradient dv = 2 (v - (x1 - x0)),
// once with the cross-entropy head gradient softmax(logits) - onehot(k1).  Weight gradients are accumulated with one thread
// per weight element looping over the live particles in ascending order, into the CTA's own slice [2][layout.total]: no
// atomics, and P depends on the dims and B only, so the bits do not depend on the device.  A jet without a live particle is
// skipped (its forward is NaN, epic.py:141, and the losses exclude it).
// epic_grad_reduce_kernel adds the P slices in slice order in fp64 and divides by the live count, read on the device.
#include "mmb_device.cuh"
#include "mmb_internal.h"

namespace mmb {

namespace {

constexpr int kThreads = 128;
constexpr int kMaxCtas = 1024;
constexpr size_t kSliceCapBytes = size_t(512) << 20;   // all P gradient slices together
constexpr size_t kHeaderBytes = (size_t)kMaxCtas * 3 * sizeof(double);

struct GradDims {
    int Dc, S, T, C, D, H, G, L, skip, Sh, X;
    int TX, K0, Kg, Kl, HW;   // T+X, local_0 / fc_global1 / fc_local1 in-widths, output width Dc+S
};

GradDims make_grad_dims(const MmbEpicDims& d) {
    GradDims f{d.dim_continuous, d.vocab_size, d.dim_time_emb, d.dim_cont_emb, d.dim_disc_emb, d.dim_hidden_local,
               d.dim_hidden_glob, d.num_blocks, d.skip_connection, d.disc_head_hidden, d.dim_context, 0, 0, 0, 0, 0};
    f.TX = f.T + f.X;
    f.K0 = f.T + f.C + f.D;
    f.Kg = 2 * f.H + f.G + f.TX;
    f.Kl = f.H + f.G + f.TX;
    f.HW = f.Dc + f.S;
    return f;
}

// Float offsets inside one CTA's region of the workspace.
struct Region {
    size_t slice;                                                      // [2][total] weight gradients (MSE, CE)
    size_t feat, a0, xl, p, q, t1, ho, z, r, lg, ls;                   // forward, per particle
    size_t dh, dz, dlg, dx, ds, dq, dp, de, dk;                        // backward, per particle
    size_t temb, pj, sum, red, pool0, g0p, g0a, g1p, g1a, xgp, xg, skg;  // forward, per jet
    size_t pool, wp, wa, up, lj;                                       // forward, per jet and layer
    size_t dxg, dsg, dpj, du, dg, dw, dpool, dctx;                     // backward, per jet
    size_t floats;
};

Region make_region(const GradDims& f, int N, size_t total) {
    Region R;
    size_t o = 0;
    auto take = [&](size_t n) { const size_t at = o; o += (n + 3) & ~size_t(3); return at; };
    const size_t n = (size_t)N, L = (size_t)f.L, H = (size_t)f.H, G = (size_t)f.G;
    R.slice = take(2 * total);
    R.feat = take(n * f.K0);
    R.a0 = take(n * H);
    R.xl = take((L + 1) * n * H);   // [L+1][N][H]: the projection's masked output, then each layer's output
    R.p = take(L * n * H);          // [L][N][H] fc_local1 pre-activation
    R.q = take(L * n * H);          // [L][N][H] fc_local2 pre-activation plus the residual
    R.t1 = take(n * H);
    R.ho = take(n * f.HW);
    R.z = take(n * (f.Sh ? f.Sh : 1));
    R.r = take(n * (f.Sh ? f.Sh : 1));
    R.lg = take(n * f.S);
    R.ls = take(n * 2);
    R.dh = take(n * f.HW);
    R.dz = take(n * (f.Sh ? f.Sh : 1));
    R.dlg = take(n * f.S);
    R.dx = take(n * H);
    R.ds = take(n * H);
    R.dq = take(n * H);
    R.dp = take(n * H);
    R.de = take(n * (f.C ? f.C : 1));
    R.dk = take(n * (f.D ? f.D : 1));
    R.temb = take(f.TX);
    R.pj = take(H);
    R.sum = take(H);
    R.red = take(4 * H);
    R.pool0 = take(2 * H + f.TX);
    R.g0p = take(H);
    R.g0a = take(H);
    R.g1p = take(H);
    R.g1a = take(H);
    R.xgp = take(G);
    R.xg = take(G);
    R.skg = take(G);
    R.pool = take(L * f.Kg);
    R.wp = take(L * H);
    R.wa = take(L * H);
    R.up = take(L * G);
    R.lj = take(L * (G + f.TX));
    R.dxg = take(G);
    R.dsg = take(G);
    R.dpj = take(H);
    R.du = take(G);
    R.dg = take(H);
    R.dw = take(H);
    R.dpool = take((size_t)f.Kg > 2 * H + f.TX ? (size_t)f.Kg : 2 * H + f.TX);
    R.dctx = take(f.X ? f.X : 1);
    R.floats = (o + 63) & ~size_t(63);
    return R;
}

int grad_ctas(const MmbEpicLayout& Lo, int B) {
    size_t cap = kSliceCapBytes / (2 * Lo.total * sizeof(float));
    cap = cap < 1 ? 1 : (cap > (size_t)kMaxCtas ? (size_t)kMaxCtas : cap);
    return (size_t)B < cap ? B : (int)cap;
}

struct GradArgs {
    const float* W;
    MmbEpicLayout Lo;
    GradDims f;
    Region R;
    const float* x;
    const uint8_t* k;
    const uint8_t* mask;
    const float* temb;
    int temb_stride;
    const float* x0;
    const float* x1;
    const uint8_t* k1;
    int B, N, P;
    float* ws;          // first CTA region
    double* part;       // [P][3] (mse, ce, live) per CTA
    float* d_context;   // [2][B][X] unscaled, nullable
    int want_grad;
};

__device__ __forceinline__ float dlrelu(float a, float d) { return a > 0.0f ? d : __fmul_rn(d, 0.01f); }
__device__ __forceinline__ float dselu(float a, float d) {
    const float scale = 1.0507009873554804934193349852946f;
    const float alpha_scale = 1.0507009873554804934193349852946f * 1.6732632423543772848170429916717f;
    return a > 0.0f ? __fmul_rn(d, scale) : __fmul_rn(d, __fmul_rn(alpha_scale, expf(a)));
}
template <int ACT>
__device__ __forceinline__ float act(float v) { return ACT == 1 ? lrelu(v) : (ACT == 2 ? selu(v) : v); }

// g[o*ldg + i] += sum over the listed particles (ascending) of dY[n*ldy + o] * act(X[n*ldx + i]); one thread per element.
// A per-jet outer product is the list {0} with ldy = ldx = 0.
template <int ACT>
__device__ void wgrad(float* g, int ldg, int O, int I, const float* dY, int ldy, const float* X, int ldx, const int* list, int cnt) {
    for (int e = threadIdx.x; e < O * I; e += kThreads) {
        const int o = e / I, i = e - o * I;
        float acc = 0.0f;
        for (int j = 0; j < cnt; ++j) {
            const size_t n = (size_t)list[j];
            acc = __fmaf_rn(dY[n * ldy + o], act<ACT>(X[n * ldx + i]), acc);
        }
        g[(size_t)o * ldg + i] = __fadd_rn(g[(size_t)o * ldg + i], acc);
    }
}
__device__ void bgrad(float* g, int O, const float* dY, int ldy, const int* list, int cnt) {
    for (int o = threadIdx.x; o < O; o += kThreads) {
        float acc = 0.0f;
        for (int j = 0; j < cnt; ++j) acc = __fadd_rn(acc, dY[(size_t)list[j] * ldy + o]);
        g[o] = __fadd_rn(g[o], acc);
    }
}

// out[i] = sum_o W[o*ldw + i] * in[o] for i < I, ascending o; one thread per i
__device__ void tmatvec(float* out, const float* __restrict__ W, int ldw, int O, int I, const float* in) {
    for (int i = threadIdx.x; i < I; i += kThreads) {
        float acc = 0.0f;
        for (int o = 0; o < O; ++o) acc = __fmaf_rn(__ldg(W + (size_t)o * ldw + i), in[o], acc);
        out[i] = acc;
    }
}

// masked column sums of rows [N][H] in the tree order of epic_fp32.cu's pooled_sums: lane partial over ascending n from +0,
// xor butterfly per warp, warps in order
__device__ void pooled_sums(const float* rows, const uint8_t* mask, int N, int H, float* red, float* sum) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int o = 0; o < H; ++o) {
        float part = 0.0f;
        for (int n = tid; n < N; n += kThreads) part = __fadd_rn(part, __fmul_rn(rows[(size_t)n * H + o], (float)mask[n]));
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) part = __fadd_rn(part, __shfl_xor_sync(0xffffffffu, part, off));
        if (lane == 0) red[warp * H + o] = part;
    }
    __syncthreads();
    for (int o = tid; o < H; o += kThreads) sum[o] = __fadd_rn(__fadd_rn(__fadd_rn(red[o], red[H + o]), red[2 * H + o]), red[3 * H + o]);
    __syncthreads();
}

struct Jet {
    const float* x;
    const uint8_t* k;
    const uint8_t* mask;
    const float* x0;
    const float* x1;
    const uint8_t* k1;
    int b, nl;
    float cnt;
};

// Forward of one jet, the IEEE operations of epic_forward_jet in the same order, activations kept in the region.
__device__ void forward_jet(const GradArgs& a, float* base, const Jet& J) {
    const float* __restrict__ W = a.W;
    const MmbEpicLayout& Lo = a.Lo;
    const GradDims& f = a.f;
    const Region& R = a.R;
    const int tid = threadIdx.x, N = a.N, H = f.H, G = f.G, T = f.T, C = f.C, D = f.D, K0 = f.K0, TX = f.TX;
    float *TEMB = base + R.temb, *PJ = base + R.pj, *SUM = base + R.sum, *RED = base + R.red;
    float *FEAT = base + R.feat, *A0 = base + R.a0, *XL = base + R.xl, *XG = base + R.xg, *SKG = base + R.skg;
    for (int i = tid; i < TX; i += kThreads) TEMB[i] = a.temb[(size_t)J.b * a.temb_stride + i];
    __syncthreads();
    for (int o = tid; o < H; o += kThreads) PJ[o] = dot_from(__ldg(W + Lo.local0_b + o), W + Lo.local0_w + (size_t)o * K0, TEMB, T);
    __syncthreads();
    // InputEmbeddings + local_0; XL[0] holds lrelu(.) unmasked here
    for (int n = tid; n < N; n += kThreads) {
        float* xn = XL + (size_t)n * H;
        if (J.mask[n]) {
            float* ft = FEAT + (size_t)n * K0;
            for (int t = 0; t < T; ++t) ft[t] = TEMB[t];
            for (int c = 0; c < C; ++c)
                ft[T + c] = dot_from(__ldg(W + Lo.emb_cont_b + c), W + Lo.emb_cont_w + (size_t)c * f.Dc, J.x + (size_t)n * f.Dc, f.Dc);
            const float* e = W + Lo.emb_disc + (size_t)J.k[n] * D;
            for (int d = 0; d < D; ++d) ft[T + C + d] = __ldg(e + d);
            for (int o = 0; o < H; ++o) {
                const float acc = dot_from(PJ[o], W + Lo.local0_w + (size_t)o * K0 + T, ft + T, C + D);
                A0[(size_t)n * H + o] = acc;
                xn[o] = lrelu(acc);
            }
        } else {
            for (int o = 0; o < H; ++o) xn[o] = lrelu(__ldg(W + Lo.local0_b + o));
        }
    }
    __syncthreads();
    // meansum_pool + global_0..2
    float *POOL0 = base + R.pool0, *G0P = base + R.g0p, *G0A = base + R.g0a, *G1P = base + R.g1p, *G1A = base + R.g1a,
          *XGP = base + R.xgp;
    pooled_sums(XL, J.mask, N, H, RED, SUM);
    for (int o = tid; o < H; o += kThreads) {
        POOL0[o] = __fdiv_rn(SUM[o], J.cnt);
        POOL0[H + o] = SUM[o];
    }
    for (int i = tid; i < TX; i += kThreads) POOL0[2 * H + i] = TEMB[i];
    __syncthreads();
    for (int o = tid; o < H; o += kThreads) {
        G0P[o] = dot_from(__ldg(W + Lo.global0_b + o), W + Lo.global0_w + (size_t)o * (2 * H + TX), POOL0, 2 * H + TX);
        G0A[o] = lrelu(G0P[o]);
    }
    __syncthreads();
    for (int o = tid; o < H; o += kThreads) {
        G1P[o] = dot_from(__ldg(W + Lo.global1_b + o), W + Lo.global1_w + (size_t)o * H, G0A, H);
        G1A[o] = lrelu(G1P[o]);
    }
    __syncthreads();
    for (int o = tid; o < G; o += kThreads) {
        XGP[o] = dot_from(__ldg(W + Lo.global2_b + o), W + Lo.global2_w + (size_t)o * H, G1A, H);
        XG[o] = SKG[o] = lrelu(XGP[o]);
    }
    for (int n = tid; n < N; n += kThreads) {
        const float m = (float)J.mask[n];
        for (int o = 0; o < H; ++o) XL[(size_t)n * H + o] = __fmul_rn(XL[(size_t)n * H + o], m);
    }
    __syncthreads();

    // EPiC layers
    for (int l = 0; l < f.L; ++l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        const float* xin = XL + (size_t)l * N * H;
        float* xout = XL + (size_t)(l + 1) * N * H;
        float *Pl = base + R.p + (size_t)l * N * H, *Ql = base + R.q + (size_t)l * N * H;
        float *pool = base + R.pool + (size_t)l * f.Kg, *wp = base + R.wp + (size_t)l * H, *wa = base + R.wa + (size_t)l * H;
        float *up = base + R.up + (size_t)l * G, *lj = base + R.lj + (size_t)l * (G + TX);
        pooled_sums(xin, J.mask, N, H, RED, SUM);
        for (int o = tid; o < H; o += kThreads) {
            pool[o] = __fdiv_rn(SUM[o], J.cnt);
            pool[H + o] = SUM[o];
        }
        for (int i = tid; i < G; i += kThreads) pool[2 * H + i] = XG[i];
        for (int i = tid; i < TX; i += kThreads) pool[2 * H + G + i] = TEMB[i];
        __syncthreads();
        for (int o = tid; o < H; o += kThreads) {
            wp[o] = dot_from(__ldg(Wl + Lo.l_g1_b + o), Wl + Lo.l_g1_w + (size_t)o * f.Kg, pool, f.Kg);
            wa[o] = lrelu(wp[o]);
        }
        __syncthreads();
        for (int o = tid; o < G; o += kThreads) {
            up[o] = __fadd_rn(dot_from(__ldg(Wl + Lo.l_g2_b + o), Wl + Lo.l_g2_w + (size_t)o * H, wa, H), XG[o]);
            lj[o] = lrelu(up[o]);   // [xg' | context]: the per-jet input of fc_local1
        }
        for (int i = tid; i < TX; i += kThreads) lj[G + i] = TEMB[i];
        __syncthreads();
        for (int o = tid; o < H; o += kThreads)
            PJ[o] = dot_from(__ldg(Wl + Lo.l_l1_b + o), Wl + Lo.l_l1_w + (size_t)o * f.Kl + H, lj, G + TX);
        __syncthreads();
        for (int n = tid; n < N; n += kThreads) {
            float* xo = xout + (size_t)n * H;
            if (!J.mask[n]) {   // a masked particle's row only ever enters a sum multiplied by its zero mask
                for (int o = 0; o < H; ++o) xo[o] = 0.0f;
                continue;
            }
            const float* xn = xin + (size_t)n * H;
            float* t1 = base + R.t1 + (size_t)n * H;
            for (int o = 0; o < H; ++o) {
                const float p = dot_from(PJ[o], Wl + Lo.l_l1_w + (size_t)o * f.Kl, xn, H);
                Pl[(size_t)n * H + o] = p;
                t1[o] = lrelu(p);
            }
            for (int o = 0; o < H; ++o) {
                const float q = __fadd_rn(dot_from(__ldg(Wl + Lo.l_l2_b + o), Wl + Lo.l_l2_w + (size_t)o * H, t1, H), xn[o]);
                Ql[(size_t)n * H + o] = q;
                float val = lrelu(q);
                if (f.skip) val = __fadd_rn(val, XL[(size_t)n * H + o]);
                xo[o] = val;
            }
        }
        for (int o = tid; o < G; o += kThreads) XG[o] = f.skip ? __fadd_rn(lj[o], SKG[o]) : lj[o];
        __syncthreads();
    }

    // output layer + heads, per-particle loss terms (the operations of bridge_losses_partial_kernel)
    for (int n = tid; n < N; n += kThreads) {
        if (!J.mask[n]) continue;
        const float* xn = XL + ((size_t)f.L * N + n) * H;
        float* h = base + R.ho + (size_t)n * f.HW;
        float* lg = base + R.lg + (size_t)n * f.S;
        for (int o = 0; o < f.HW; ++o) h[o] = dot_from(__ldg(W + Lo.out_b + o), W + Lo.out_w + (size_t)o * H, xn, H);
        if (f.Sh) {
            float *z = base + R.z + (size_t)n * f.Sh, *r = base + R.r + (size_t)n * f.Sh;
            for (int o = 0; o < f.Sh; ++o) {
                z[o] = dot_from(__ldg(W + Lo.head0_b + o), W + Lo.head0_w + (size_t)o * f.S, h + f.Dc, f.S);
                r[o] = selu(z[o]);
            }
            for (int o = 0; o < f.S; ++o) lg[o] = dot_from(__ldg(W + Lo.head2_b + o), W + Lo.head2_w + (size_t)o * f.Sh, r, f.Sh);
        } else {
            for (int o = 0; o < f.S; ++o) lg[o] = h[f.Dc + o];
        }
        float e = 0.0f;
        for (int c = 0; c < f.Dc; ++c) {
            const float d = h[c] - (J.x1[(size_t)n * f.Dc + c] - J.x0[(size_t)n * f.Dc + c]);
            e = fmaf(d, d, e);
        }
        float mx = -INFINITY;
        for (int s = 0; s < f.S; ++s) mx = fmaxf(mx, lg[s]);
        float se = 0.0f;
        for (int s = 0; s < f.S; ++s) se += expf(lg[s] - mx);
        base[R.ls + 2 * n] = e;
        base[R.ls + 2 * n + 1] = (mx + logf(se)) - lg[J.k1[n]];
    }
    __syncthreads();
}

// Backward of one jet for one loss (which = 0: MSE, 1: CE), unnormalised, into slice `which` of the CTA.
__device__ void backward_jet(const GradArgs& a, float* base, const Jet& J, const int* live, const int* one, int which) {
    const float* __restrict__ W = a.W;
    const MmbEpicLayout& Lo = a.Lo;
    const GradDims& f = a.f;
    const Region& R = a.R;
    const int tid = threadIdx.x, N = a.N, H = f.H, G = f.G, T = f.T, TX = f.TX, nl = J.nl;
    float* gw = base + R.slice + (size_t)which * Lo.total;
    float *DH = base + R.dh, *DZ = base + R.dz, *DLG = base + R.dlg, *DX = base + R.dx, *DS = base + R.ds, *DQ = base + R.dq,
          *DP = base + R.dp;
    float *DXG = base + R.dxg, *DSG = base + R.dsg, *DPJ = base + R.dpj, *DU = base + R.du, *DG = base + R.dg, *DW = base + R.dw,
          *DPOOL = base + R.dpool, *DCTX = base + R.dctx;
    const float* XL = base + R.xl;

    // head gradients -> dh -> d(last local hidden)
    for (int n = tid; n < N; n += kThreads) {
        if (!J.mask[n]) continue;
        const float* h = base + R.ho + (size_t)n * f.HW;
        const float* lg = base + R.lg + (size_t)n * f.S;
        float* dh = DH + (size_t)n * f.HW;
        if (which == 0) {
            for (int c = 0; c < f.Dc; ++c)
                dh[c] = __fmul_rn(2.0f, h[c] - (J.x1[(size_t)n * f.Dc + c] - J.x0[(size_t)n * f.Dc + c]));
            for (int s = 0; s < f.S; ++s) dh[f.Dc + s] = 0.0f;
        } else {
            for (int c = 0; c < f.Dc; ++c) dh[c] = 0.0f;
            float mx = -INFINITY;
            for (int s = 0; s < f.S; ++s) mx = fmaxf(mx, lg[s]);
            float se = 0.0f;
            for (int s = 0; s < f.S; ++s) se += expf(lg[s] - mx);
            float* dl = f.Sh ? DLG + (size_t)n * f.S : dh + f.Dc;
            for (int s = 0; s < f.S; ++s) dl[s] = __fdiv_rn(expf(lg[s] - mx), se) - (s == J.k1[n] ? 1.0f : 0.0f);
            if (f.Sh) {
                const float* z = base + R.z + (size_t)n * f.Sh;
                float* dz = DZ + (size_t)n * f.Sh;
                for (int o = 0; o < f.Sh; ++o) {
                    float acc = 0.0f;
                    for (int s = 0; s < f.S; ++s) acc = __fmaf_rn(__ldg(W + Lo.head2_w + (size_t)s * f.Sh + o), dl[s], acc);
                    dz[o] = dselu(z[o], acc);
                }
                for (int s = 0; s < f.S; ++s) {
                    float acc = 0.0f;
                    for (int o = 0; o < f.Sh; ++o) acc = __fmaf_rn(__ldg(W + Lo.head0_w + (size_t)o * f.S + s), dz[o], acc);
                    dh[f.Dc + s] = acc;
                }
            }
        }
        float* dx = DX + (size_t)n * H;
        for (int i = 0; i < H; ++i) {
            float acc = 0.0f;
            for (int o = 0; o < f.HW; ++o) acc = __fmaf_rn(__ldg(W + Lo.out_w + (size_t)o * H + i), dh[o], acc);
            dx[i] = acc;
            DS[(size_t)n * H + i] = 0.0f;
        }
    }
    for (int g = tid; g < G; g += kThreads) DXG[g] = DSG[g] = 0.0f;
    for (int i = tid; i < f.X; i += kThreads) DCTX[i] = 0.0f;
    __syncthreads();
    wgrad<0>(gw + Lo.out_w, H, f.HW, H, DH, f.HW, XL + (size_t)f.L * N * H, H, live, nl);
    bgrad(gw + Lo.out_b, f.HW, DH, f.HW, live, nl);
    if (which == 1 && f.Sh) {
        wgrad<2>(gw + Lo.head2_w, f.Sh, f.S, f.Sh, DLG, f.S, base + R.z, f.Sh, live, nl);
        bgrad(gw + Lo.head2_b, f.S, DLG, f.S, live, nl);
        wgrad<0>(gw + Lo.head0_w, f.S, f.Sh, f.S, DZ, f.Sh, base + R.ho + f.Dc, f.HW, live, nl);
        bgrad(gw + Lo.head0_b, f.Sh, DZ, f.Sh, live, nl);
    }
    __syncthreads();

    // EPiC layers, last to first
    for (int l = f.L - 1; l >= 0; --l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        float* gl = gw + Lo.layer0 + (size_t)l * Lo.layer_stride;
        const float *xin = XL + (size_t)l * N * H, *Pl = base + R.p + (size_t)l * N * H, *Ql = base + R.q + (size_t)l * N * H;
        const float *pool = base + R.pool + (size_t)l * f.Kg, *wp = base + R.wp + (size_t)l * H, *up = base + R.up + (size_t)l * G;
        const float* lj = base + R.lj + (size_t)l * (G + TX);
        // fc_local2 (+ residual, skip) and fc_local1, per live particle
        for (int n = tid; n < N; n += kThreads) {
            if (!J.mask[n]) continue;
            float *dx = DX + (size_t)n * H, *ds = DS + (size_t)n * H, *dq = DQ + (size_t)n * H, *dp = DP + (size_t)n * H;
            const float *q = Ql + (size_t)n * H, *p = Pl + (size_t)n * H;
            for (int o = 0; o < H; ++o) {
                if (f.skip) ds[o] = __fadd_rn(ds[o], dx[o]);
                dq[o] = dlrelu(q[o], dx[o]);
            }
            for (int i = 0; i < H; ++i) {
                float acc = 0.0f;
                for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(Wl + Lo.l_l2_w + (size_t)o * H + i), dq[o], acc);
                dp[i] = dlrelu(p[i], acc);
            }
            for (int i = 0; i < H; ++i) {
                float acc = dq[i];
                for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(Wl + Lo.l_l1_w + (size_t)o * f.Kl + i), dp[o], acc);
                dx[i] = acc;
            }
        }
        __syncthreads();
        // per-jet chain: fc_local1's jet columns, fc_global2 (+ residual), fc_global1, pooling
        for (int o = tid; o < H; o += kThreads) {
            float acc = 0.0f;
            for (int j = 0; j < nl; ++j) acc = __fadd_rn(acc, DP[(size_t)live[j] * H + o]);
            DPJ[o] = acc;
        }
        if (f.skip)
            for (int g = tid; g < G; g += kThreads) DSG[g] = __fadd_rn(DSG[g], DXG[g]);
        __syncthreads();
        for (int g = tid; g < G; g += kThreads) {
            float acc = DXG[g];
            for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(Wl + Lo.l_l1_w + (size_t)o * f.Kl + H + g), DPJ[o], acc);
            DU[g] = dlrelu(up[g], acc);
        }
        for (int i = tid; i < f.X; i += kThreads) {
            float acc = 0.0f;
            for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(Wl + Lo.l_l1_w + (size_t)o * f.Kl + H + G + T + i), DPJ[o], acc);
            DCTX[i] = __fadd_rn(DCTX[i], acc);
        }
        __syncthreads();
        for (int h = tid; h < H; h += kThreads) {
            float acc = 0.0f;
            for (int g = 0; g < G; ++g) acc = __fmaf_rn(__ldg(Wl + Lo.l_g2_w + (size_t)g * H + h), DU[g], acc);
            DW[h] = dlrelu(wp[h], acc);
        }
        __syncthreads();
        tmatvec(DPOOL, Wl + Lo.l_g1_w, f.Kg, H, f.Kg, DW);
        __syncthreads();
        for (int g = tid; g < G; g += kThreads) DXG[g] = __fadd_rn(DU[g], DPOOL[2 * H + g]);
        for (int i = tid; i < f.X; i += kThreads) DCTX[i] = __fadd_rn(DCTX[i], DPOOL[2 * H + G + T + i]);
        for (int n = tid; n < N; n += kThreads) {   // masked mean + sum pooling: dmean / cnt + dsum
            if (!J.mask[n]) continue;
            float* dx = DX + (size_t)n * H;
            for (int i = 0; i < H; ++i) dx[i] = __fadd_rn(dx[i], __fadd_rn(__fdiv_rn(DPOOL[i], J.cnt), DPOOL[H + i]));
        }
        wgrad<1>(gl + Lo.l_l2_w, H, H, H, DQ, H, Pl, H, live, nl);
        bgrad(gl + Lo.l_l2_b, H, DQ, H, live, nl);
        wgrad<0>(gl + Lo.l_l1_w, f.Kl, H, H, DP, H, xin, H, live, nl);
        wgrad<0>(gl + Lo.l_l1_w + H, f.Kl, H, G + TX, DPJ, 0, lj, 0, one, 1);
        bgrad(gl + Lo.l_l1_b, H, DPJ, 0, one, 1);
        wgrad<1>(gl + Lo.l_g2_w, H, G, H, DU, 0, wp, 0, one, 1);
        bgrad(gl + Lo.l_g2_b, G, DU, 0, one, 1);
        wgrad<0>(gl + Lo.l_g1_w, f.Kg, H, f.Kg, DW, 0, pool, 0, one, 1);
        bgrad(gl + Lo.l_g1_b, H, DW, 0, one, 1);
        __syncthreads();
    }

    // projection: global_2..0, pooling, local_0, the embeddings
    const float *G0P = base + R.g0p, *G1P = base + R.g1p, *XGP = base + R.xgp;
    for (int g = tid; g < G; g += kThreads) DU[g] = dlrelu(XGP[g], __fadd_rn(DXG[g], DSG[g]));
    __syncthreads();
    for (int h = tid; h < H; h += kThreads) {
        float acc = 0.0f;
        for (int g = 0; g < G; ++g) acc = __fmaf_rn(__ldg(W + Lo.global2_w + (size_t)g * H + h), DU[g], acc);
        DW[h] = dlrelu(G1P[h], acc);
    }
    __syncthreads();
    for (int h = tid; h < H; h += kThreads) {
        float acc = 0.0f;
        for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(W + Lo.global1_w + (size_t)o * H + h), DW[o], acc);
        DG[h] = dlrelu(G0P[h], acc);
    }
    __syncthreads();
    tmatvec(DPOOL, W + Lo.global0_w, 2 * H + TX, H, 2 * H + TX, DG);
    __syncthreads();
    for (int i = tid; i < f.X; i += kThreads) DCTX[i] = __fadd_rn(DCTX[i], DPOOL[2 * H + T + i]);
    const int C = f.C, D = f.D, K0 = f.K0;
    float *DE = base + R.de, *DK = base + R.dk;
    for (int n = tid; n < N; n += kThreads) {
        if (!J.mask[n]) continue;
        const float* a0 = base + R.a0 + (size_t)n * H;
        const float *dx = DX + (size_t)n * H, *ds = DS + (size_t)n * H;
        float* da = DQ + (size_t)n * H;
        for (int o = 0; o < H; ++o) {
            float d = __fadd_rn(dx[o], __fadd_rn(__fdiv_rn(DPOOL[o], J.cnt), DPOOL[H + o]));
            if (f.skip) d = __fadd_rn(d, ds[o]);
            da[o] = dlrelu(a0[o], d);
        }
        for (int c = 0; c < C; ++c) {
            float acc = 0.0f;
            for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(W + Lo.local0_w + (size_t)o * K0 + T + c), da[o], acc);
            DE[(size_t)n * C + c] = acc;
        }
        for (int d = 0; d < D; ++d) {
            float acc = 0.0f;
            for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(W + Lo.local0_w + (size_t)o * K0 + T + C + d), da[o], acc);
            DK[(size_t)n * D + d] = acc;
        }
    }
    __syncthreads();
    wgrad<1>(gw + Lo.global2_w, H, G, H, DU, 0, G1P, 0, one, 1);
    bgrad(gw + Lo.global2_b, G, DU, 0, one, 1);
    wgrad<1>(gw + Lo.global1_w, H, H, H, DW, 0, G0P, 0, one, 1);
    bgrad(gw + Lo.global1_b, H, DW, 0, one, 1);
    wgrad<0>(gw + Lo.global0_w, 2 * H + TX, H, 2 * H + TX, DG, 0, base + R.pool0, 0, one, 1);
    bgrad(gw + Lo.global0_b, H, DG, 0, one, 1);
    wgrad<0>(gw + Lo.local0_w, K0, H, K0, DQ, H, base + R.feat, K0, live, nl);
    bgrad(gw + Lo.local0_b, H, DQ, H, live, nl);
    wgrad<0>(gw + Lo.emb_cont_w, f.Dc, C, f.Dc, DE, C, J.x, f.Dc, live, nl);
    bgrad(gw + Lo.emb_cont_b, C, DE, C, live, nl);
    for (int e = tid; e < f.S * D; e += kThreads) {   // embedding table: rows scattered by token, particles ascending
        const int s = e / D, d = e - s * D;
        float acc = 0.0f;
        for (int j = 0; j < nl; ++j)
            if (J.k[live[j]] == s) acc = __fadd_rn(acc, DK[(size_t)live[j] * D + d]);
        gw[Lo.emb_disc + e] = __fadd_rn(gw[Lo.emb_disc + e], acc);
    }
    if (a.d_context)
        for (int i = tid; i < f.X; i += kThreads) a.d_context[((size_t)which * a.B + J.b) * f.X + i] = DCTX[i];
    __syncthreads();
}

__global__ void __launch_bounds__(kThreads) epic_loss_grad_kernel(GradArgs a) {
    extern __shared__ int s_live[];   // [N] live particles of the current jet, ascending
    __shared__ int s_n, s_one;
    __shared__ double s_acc[3];
    const int tid = threadIdx.x, N = a.N;
    float* base = a.ws + (size_t)blockIdx.x * a.R.floats;
    if (a.want_grad)
        for (size_t e = tid; e < 2 * a.Lo.total; e += kThreads) base[a.R.slice + e] = 0.0f;
    if (tid == 0) {
        s_one = 0;
        s_acc[0] = s_acc[1] = s_acc[2] = 0.0;
    }
    for (int b = blockIdx.x; b < a.B; b += a.P) {
        const uint8_t* mask = a.mask + (size_t)b * N;
        __syncthreads();
        if (tid == 0) {
            int c = 0;
            for (int n = 0; n < N; ++n)
                if (mask[n]) s_live[c++] = n;
            s_n = c;
        }
        __syncthreads();
        const int nl = s_n;
        if (nl == 0) {   // no gradient reaches the context of an empty jet
            if (a.d_context)
                for (int i = tid; i < 2 * a.f.X; i += kThreads) a.d_context[((size_t)(i / a.f.X) * a.B + b) * a.f.X + i % a.f.X] = 0.0f;
            continue;
        }
        const Jet J{a.x + (size_t)b * N * a.f.Dc, a.k + (size_t)b * N, mask, a.x0 + (size_t)b * N * a.f.Dc, a.x1 + (size_t)b * N * a.f.Dc,
                    a.k1 + (size_t)b * N, b, nl, (float)nl};
        forward_jet(a, base, J);
        if (tid == 0) {
            for (int j = 0; j < nl; ++j) {
                s_acc[0] += (double)base[a.R.ls + 2 * s_live[j]];
                s_acc[1] += (double)base[a.R.ls + 2 * s_live[j] + 1];
            }
            s_acc[2] += (double)nl;
        }
        if (a.want_grad) {
            backward_jet(a, base, J, s_live, &s_one, 0);
            backward_jet(a, base, J, s_live, &s_one, 1);
        }
    }
    __syncthreads();
    if (tid < 3) a.part[(size_t)blockIdx.x * 3 + tid] = s_acc[tid];
}

// losses = {mse, ce, live}; jac[e] = sum_p slice_p[e] / live in fp64, slices in order; d_context scaled by 1 / live in place
__global__ void __launch_bounds__(256) epic_grad_reduce_kernel(const float* __restrict__ ws, size_t region_floats, size_t slice_off,
                                                               const double* __restrict__ part, int P, size_t n_jac, float* __restrict__ jac,
                                                               float* d_context, size_t n_ctx, float* __restrict__ losses) {
    __shared__ double s_live;
    if (threadIdx.x == 0) {
        double m = 0, c = 0, n = 0;
        for (int p = 0; p < P; ++p) {
            m += part[(size_t)p * 3];
            c += part[(size_t)p * 3 + 1];
            n += part[(size_t)p * 3 + 2];
        }
        s_live = n;
        if (blockIdx.x == 0) {
            losses[0] = (float)(m / n);
            losses[1] = (float)(c / n);
            losses[2] = (float)n;
        }
    }
    __syncthreads();
    const double live = s_live;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_jac + n_ctx; e += (size_t)gridDim.x * blockDim.x) {
        if (e < n_jac) {
            double acc = 0.0;
            for (int p = 0; p < P; ++p) acc += (double)ws[(size_t)p * region_floats + slice_off + e];
            jac[e] = (float)(acc / live);
        } else {
            d_context[e - n_jac] = (float)((double)d_context[e - n_jac] / live);
        }
    }
}

}  // namespace

size_t epic_loss_grad_workspace_bytes(const MmbEpicDims& d, int B, int N) {
    const MmbEpicLayout Lo = mmb_epic_layout(&d);
    const Region R = make_region(make_grad_dims(d), N, Lo.total);
    return kHeaderBytes + (size_t)grad_ctas(Lo, B) * R.floats * sizeof(float);
}

int launch_epic_loss_grad(const MmbEpicDims& d, const float* W, const float* x, const uint8_t* k, const uint8_t* mask, const float* temb,
                          int temb_stride, const float* x0, const float* x1, const uint8_t* k1, int B, int N, float* losses, float* jac,
                          float* d_context, void* workspace, cudaStream_t stream) {
    GradArgs a;
    a.W = W;
    a.Lo = mmb_epic_layout(&d);
    a.f = make_grad_dims(d);
    a.R = make_region(a.f, N, a.Lo.total);
    a.x = x, a.k = k, a.mask = mask, a.temb = temb, a.temb_stride = temb_stride;
    a.x0 = x0, a.x1 = x1, a.k1 = k1;
    a.B = B, a.N = N, a.P = grad_ctas(a.Lo, B);
    a.part = static_cast<double*>(workspace);
    a.ws = reinterpret_cast<float*>(static_cast<char*>(workspace) + kHeaderBytes);
    a.want_grad = jac != nullptr;
    a.d_context = (jac && a.f.X) ? d_context : nullptr;
    epic_loss_grad_kernel<<<a.P, kThreads, (size_t)N * sizeof(int), stream>>>(a);
    if (int rc = cuda_ok(cudaGetLastError(), "epic_loss_grad launch")) return rc;
    const size_t n_jac = jac ? 2 * a.Lo.total : 0, n_ctx = a.d_context ? (size_t)2 * B * a.f.X : 0;
    const size_t want = (n_jac + n_ctx + 255) / 256;
    const unsigned blocks = (unsigned)(want < 1 ? 1 : (want > 4096 ? 4096 : want));
    epic_grad_reduce_kernel<<<blocks, 256, 0, stream>>>(a.ws, a.R.floats, a.R.slice, a.part, a.P, n_jac, jac, a.d_context, n_ctx, losses);
    return cuda_ok(cudaGetLastError(), "epic_grad_reduce launch");
}

}  // namespace mmb
