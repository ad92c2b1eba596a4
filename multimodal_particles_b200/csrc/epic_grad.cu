// epic_grad.cu — the bridge-matching losses of MultiModalBridgeMatching and their gradients with respect to every weight of
// the packed EPiC blob, fp32 on CUDA cores (mbm.py:167-197, 232-240; epic.py:136-241; utils.py:112-172).
//
// epic_loss_grad_kernel: a persistent grid of P CTAs of 128 threads; CTA c takes jets c, c+P, ... in ascending order.  Per jet
// it runs the fp32 forward of mmb_epic_forward (epic_forward_jet, epic_fp32.cuh) with every activation the backward needs kept
// in the CTA's region of the workspace (Fp32Record), forms the per-particle loss terms of bridge_losses_partial_kernel
// (bridge_loss_terms), and runs the backward twice: once seeded with the MSE head gradient dv = 2 (v - (x1 - x0)),
// once with the cross-entropy head gradient softmax(logits) - onehot(k1).  Weight gradients are accumulated with one thread
// per weight element looping over the live particles in ascending order, into the CTA's own slice [2][layout.total]: no
// atomics, and P depends on the dims and B only, so the bits do not depend on the device.  A jet without a live particle is
// skipped (its forward is NaN, epic.py:141, and the losses exclude it).
// epic_grad_reduce_kernel adds the P slices in slice order in fp64 and divides by the live count, read on the device.
#include "epic_fp32.cuh"

namespace mmb {

namespace {

constexpr int kMaxCtas = 1024;
constexpr size_t kSliceCapBytes = size_t(512) << 20;   // all P gradient slices together
constexpr size_t kHeaderBytes = (size_t)kMaxCtas * 3 * sizeof(double);

// Float offsets inside one CTA's region of the workspace.
struct Region {
    size_t slice;                                                      // [2][total] weight gradients (MSE, CE)
    size_t feat, a0, xl, p, q, t1, ho, z, r, lg, ls;                   // forward, per particle
    size_t dh, dz, dlg, dx, ds, dq, dp, de, dk;                        // backward, per particle
    size_t temb, pj, sum, red, pool0, g0p, g0a, g1p, g1a, xgp, xg, skg;  // forward, per jet
    size_t pool, wp, up, lj;                                           // forward, per jet and layer
    size_t dxg, dsg, dpj, du, dg, dw, dpool, dctx;                     // backward, per jet
    size_t floats;
};

Region make_region(const Fp32Dims& f, int N, size_t total) {
    Region R;
    size_t o = 0;
    auto take = [&](size_t n) { const size_t at = o; o += (n + 3) & ~size_t(3); return at; };
    const size_t n = (size_t)N, L = (size_t)f.L, H = (size_t)f.H, G = (size_t)f.G, HW = (size_t)(f.Dc + f.S);
    R.slice = take(2 * total);
    R.feat = take(n * f.K0());
    R.a0 = take(n * H);
    R.xl = take((L + 1) * n * H);   // [L+1][N][H]: the projection's masked output, then each layer's output
    R.p = take(L * n * H);          // [L][N][H] fc_local1 pre-activation
    R.q = take(L * n * H);          // [L][N][H] fc_local2 pre-activation plus the residual
    R.t1 = take(n * H);
    R.ho = take(n * HW);
    R.z = take(n * (f.Sh ? f.Sh : 1));
    R.r = take(n * (f.Sh ? f.Sh : 1));
    R.lg = take(n * f.S);
    R.ls = take(n * 2);
    R.dh = take(n * HW);
    R.dz = take(n * (f.Sh ? f.Sh : 1));
    R.dlg = take(n * f.S);
    R.dx = take(n * H);
    R.ds = take(n * H);
    R.dq = take(n * H);
    R.dp = take(n * H);
    R.de = take(n * (f.C ? f.C : 1));
    R.dk = take(n * (f.D ? f.D : 1));
    R.temb = take(f.TX());
    R.pj = take(H);
    R.sum = take(H);
    R.red = take(4 * H);
    R.pool0 = take(2 * H + f.TX());
    R.g0p = take(H);
    R.g0a = take(H);
    R.g1p = take(H);
    R.g1a = take(H);
    R.xgp = take(G);
    R.xg = take(G);
    R.skg = take(G);
    R.pool = take(L * f.Kg());
    R.wp = take(L * H);
    R.up = take(L * G);
    R.lj = take(L * (G + f.TX()));
    R.dxg = take(G);
    R.dsg = take(G);
    R.dpj = take(H);
    R.du = take(G);
    R.dg = take(H);
    R.dw = take(H);
    R.dpool = take((size_t)f.Kg() > 2 * H + f.TX() ? (size_t)f.Kg() : 2 * H + f.TX());
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
    Fp32Dims f;
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
    for (int e = threadIdx.x; e < O * I; e += kFp32Threads) {
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
    for (int o = threadIdx.x; o < O; o += kFp32Threads) {
        float acc = 0.0f;
        for (int j = 0; j < cnt; ++j) acc = __fadd_rn(acc, dY[(size_t)list[j] * ldy + o]);
        g[o] = __fadd_rn(g[o], acc);
    }
}

// out[i] = sum_o W[o*ldw + i] * in[o] for i < I, ascending o; one thread per i
__device__ void tmatvec(float* out, const float* __restrict__ W, int ldw, int O, int I, const float* in) {
    for (int i = threadIdx.x; i < I; i += kFp32Threads) {
        float acc = 0.0f;
        for (int o = 0; o < O; ++o) acc = __fmaf_rn(__ldg(W + (size_t)o * ldw + i), in[o], acc);
        out[i] = acc;
    }
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

// Forward of one jet, its activations kept in the region, and its per-particle loss terms.
__device__ void forward_jet(const GradArgs& a, float* base, int* cnt, const Jet& J) {
    const Fp32Dims& f = a.f;
    const Region& R = a.R;
    const int tid = threadIdx.x;
    Fp32Record s;
    s.temb = base + R.temb, s.pj = base + R.pj, s.pool = base + R.pool0, s.g0 = base + R.g0a, s.g1 = base + R.g1a;
    s.xg = base + R.xg, s.skipg = base + R.skg, s.sum = base + R.sum, s.red = base + R.red, s.cnt = cnt;
    s.xl = s.skipl = base + R.xl, s.row = base + R.t1;
    s.feat = base + R.feat, s.a0 = base + R.a0, s.g0p = base + R.g0p, s.g1p = base + R.g1p, s.xgp = base + R.xgp;
    s.lpool = base + R.pool, s.wp = base + R.wp, s.up = base + R.up, s.lj = base + R.lj, s.p = base + R.p, s.q = base + R.q;
    s.ho = base + R.ho, s.z = base + R.z, s.r = base + R.r;
    for (int i = tid; i < f.TX(); i += kFp32Threads) s.temb[i] = a.temb[(size_t)J.b * a.temb_stride + i];
    __syncthreads();
    epic_forward_jet(a.W, a.Lo, f, s, J.x, J.k, J.mask, a.N, nullptr, base + R.lg, nullptr);
    for (int n = tid; n < a.N; n += kFp32Threads)   // the heads of particle n were written by this thread
        if (J.mask[n]) {
            const float2 t = bridge_loss_terms(s.ho + (size_t)n * (f.Dc + f.S), J.x0 + (size_t)n * f.Dc, J.x1 + (size_t)n * f.Dc, f.Dc,
                                               base + R.lg + (size_t)n * f.S, f.S, J.k1[n]);
            base[R.ls + 2 * n] = t.x;
            base[R.ls + 2 * n + 1] = t.y;
        }
    __syncthreads();
}

// Backward of one jet for one loss (which = 0: MSE, 1: CE), unnormalised, into slice `which` of the CTA.
__device__ void backward_jet(const GradArgs& a, float* base, const Jet& J, const int* live, const int* one, int which) {
    const float* __restrict__ W = a.W;
    const MmbEpicLayout& Lo = a.Lo;
    const Fp32Dims& f = a.f;
    const Region& R = a.R;
    const int tid = threadIdx.x, N = a.N, H = f.H, G = f.G, T = f.T, TX = f.TX(), Kg = f.Kg(), Kl = f.Kl(), HW = f.Dc + f.S,
              nl = J.nl;
    float* gw = base + R.slice + (size_t)which * Lo.total;
    float *DH = base + R.dh, *DZ = base + R.dz, *DLG = base + R.dlg, *DX = base + R.dx, *DS = base + R.ds, *DQ = base + R.dq,
          *DP = base + R.dp;
    float *DXG = base + R.dxg, *DSG = base + R.dsg, *DPJ = base + R.dpj, *DU = base + R.du, *DG = base + R.dg, *DW = base + R.dw,
          *DPOOL = base + R.dpool, *DCTX = base + R.dctx;
    const float* XL = base + R.xl;

    // head gradients -> dh -> d(last local hidden)
    for (int n = tid; n < N; n += kFp32Threads) {
        if (!J.mask[n]) continue;
        const float* h = base + R.ho + (size_t)n * HW;
        const float* lg = base + R.lg + (size_t)n * f.S;
        float* dh = DH + (size_t)n * HW;
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
            for (int o = 0; o < HW; ++o) acc = __fmaf_rn(__ldg(W + Lo.out_w + (size_t)o * H + i), dh[o], acc);
            dx[i] = acc;
            DS[(size_t)n * H + i] = 0.0f;
        }
    }
    for (int g = tid; g < G; g += kFp32Threads) DXG[g] = DSG[g] = 0.0f;
    for (int i = tid; i < f.X; i += kFp32Threads) DCTX[i] = 0.0f;
    __syncthreads();
    wgrad<0>(gw + Lo.out_w, H, HW, H, DH, HW, XL + (size_t)f.L * N * H, H, live, nl);
    bgrad(gw + Lo.out_b, HW, DH, HW, live, nl);
    if (which == 1 && f.Sh) {
        wgrad<2>(gw + Lo.head2_w, f.Sh, f.S, f.Sh, DLG, f.S, base + R.z, f.Sh, live, nl);
        bgrad(gw + Lo.head2_b, f.S, DLG, f.S, live, nl);
        wgrad<0>(gw + Lo.head0_w, f.S, f.Sh, f.S, DZ, f.Sh, base + R.ho + f.Dc, HW, live, nl);
        bgrad(gw + Lo.head0_b, f.Sh, DZ, f.Sh, live, nl);
    }
    __syncthreads();

    // EPiC layers, last to first
    for (int l = f.L - 1; l >= 0; --l) {
        const float* Wl = W + Lo.layer0 + (size_t)l * Lo.layer_stride;
        float* gl = gw + Lo.layer0 + (size_t)l * Lo.layer_stride;
        const float *xin = XL + (size_t)l * N * H, *Pl = base + R.p + (size_t)l * N * H, *Ql = base + R.q + (size_t)l * N * H;
        const float *pool = base + R.pool + (size_t)l * Kg, *wp = base + R.wp + (size_t)l * H, *up = base + R.up + (size_t)l * G;
        const float* lj = base + R.lj + (size_t)l * (G + TX);
        // fc_local2 (+ residual, skip) and fc_local1, per live particle
        for (int n = tid; n < N; n += kFp32Threads) {
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
                for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(Wl + Lo.l_l1_w + (size_t)o * Kl + i), dp[o], acc);
                dx[i] = acc;
            }
        }
        __syncthreads();
        // per-jet chain: fc_local1's jet columns, fc_global2 (+ residual), fc_global1, pooling
        for (int o = tid; o < H; o += kFp32Threads) {
            float acc = 0.0f;
            for (int j = 0; j < nl; ++j) acc = __fadd_rn(acc, DP[(size_t)live[j] * H + o]);
            DPJ[o] = acc;
        }
        if (f.skip)
            for (int g = tid; g < G; g += kFp32Threads) DSG[g] = __fadd_rn(DSG[g], DXG[g]);
        __syncthreads();
        for (int g = tid; g < G; g += kFp32Threads) {
            float acc = DXG[g];
            for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(Wl + Lo.l_l1_w + (size_t)o * Kl + H + g), DPJ[o], acc);
            DU[g] = dlrelu(up[g], acc);
        }
        for (int i = tid; i < f.X; i += kFp32Threads) {
            float acc = 0.0f;
            for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(Wl + Lo.l_l1_w + (size_t)o * Kl + H + G + T + i), DPJ[o], acc);
            DCTX[i] = __fadd_rn(DCTX[i], acc);
        }
        __syncthreads();
        for (int h = tid; h < H; h += kFp32Threads) {
            float acc = 0.0f;
            for (int g = 0; g < G; ++g) acc = __fmaf_rn(__ldg(Wl + Lo.l_g2_w + (size_t)g * H + h), DU[g], acc);
            DW[h] = dlrelu(wp[h], acc);
        }
        __syncthreads();
        tmatvec(DPOOL, Wl + Lo.l_g1_w, Kg, H, Kg, DW);
        __syncthreads();
        for (int g = tid; g < G; g += kFp32Threads) DXG[g] = __fadd_rn(DU[g], DPOOL[2 * H + g]);
        for (int i = tid; i < f.X; i += kFp32Threads) DCTX[i] = __fadd_rn(DCTX[i], DPOOL[2 * H + G + T + i]);
        for (int n = tid; n < N; n += kFp32Threads) {   // masked mean + sum pooling: dmean / cnt + dsum
            if (!J.mask[n]) continue;
            float* dx = DX + (size_t)n * H;
            for (int i = 0; i < H; ++i) dx[i] = __fadd_rn(dx[i], __fadd_rn(__fdiv_rn(DPOOL[i], J.cnt), DPOOL[H + i]));
        }
        wgrad<1>(gl + Lo.l_l2_w, H, H, H, DQ, H, Pl, H, live, nl);
        bgrad(gl + Lo.l_l2_b, H, DQ, H, live, nl);
        wgrad<0>(gl + Lo.l_l1_w, Kl, H, H, DP, H, xin, H, live, nl);
        wgrad<0>(gl + Lo.l_l1_w + H, Kl, H, G + TX, DPJ, 0, lj, 0, one, 1);
        bgrad(gl + Lo.l_l1_b, H, DPJ, 0, one, 1);
        wgrad<1>(gl + Lo.l_g2_w, H, G, H, DU, 0, wp, 0, one, 1);
        bgrad(gl + Lo.l_g2_b, G, DU, 0, one, 1);
        wgrad<0>(gl + Lo.l_g1_w, Kg, H, Kg, DW, 0, pool, 0, one, 1);
        bgrad(gl + Lo.l_g1_b, H, DW, 0, one, 1);
        __syncthreads();
    }

    // projection: global_2..0, pooling, local_0, the embeddings
    const float *G0P = base + R.g0p, *G1P = base + R.g1p, *XGP = base + R.xgp;
    for (int g = tid; g < G; g += kFp32Threads) DU[g] = dlrelu(XGP[g], __fadd_rn(DXG[g], DSG[g]));
    __syncthreads();
    for (int h = tid; h < H; h += kFp32Threads) {
        float acc = 0.0f;
        for (int g = 0; g < G; ++g) acc = __fmaf_rn(__ldg(W + Lo.global2_w + (size_t)g * H + h), DU[g], acc);
        DW[h] = dlrelu(G1P[h], acc);
    }
    __syncthreads();
    for (int h = tid; h < H; h += kFp32Threads) {
        float acc = 0.0f;
        for (int o = 0; o < H; ++o) acc = __fmaf_rn(__ldg(W + Lo.global1_w + (size_t)o * H + h), DW[o], acc);
        DG[h] = dlrelu(G0P[h], acc);
    }
    __syncthreads();
    tmatvec(DPOOL, W + Lo.global0_w, 2 * H + TX, H, 2 * H + TX, DG);
    __syncthreads();
    for (int i = tid; i < f.X; i += kFp32Threads) DCTX[i] = __fadd_rn(DCTX[i], DPOOL[2 * H + T + i]);
    const int C = f.C, D = f.D, K0 = f.K0();
    float *DE = base + R.de, *DK = base + R.dk;
    for (int n = tid; n < N; n += kFp32Threads) {
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
    for (int e = tid; e < f.S * D; e += kFp32Threads) {   // embedding table: rows scattered by token, particles ascending
        const int s = e / D, d = e - s * D;
        float acc = 0.0f;
        for (int j = 0; j < nl; ++j)
            if (J.k[live[j]] == s) acc = __fadd_rn(acc, DK[(size_t)live[j] * D + d]);
        gw[Lo.emb_disc + e] = __fadd_rn(gw[Lo.emb_disc + e], acc);
    }
    if (a.d_context)
        for (int i = tid; i < f.X; i += kFp32Threads) a.d_context[((size_t)which * a.B + J.b) * f.X + i] = DCTX[i];
    __syncthreads();
}

// No minimum-CTAs bound: holding the kernel to 72 registers (7 CTAs per SM) measured slower at the C2 widths, B = 4096 (DESIGN.md §4.8).
__global__ void __launch_bounds__(kFp32Threads) epic_loss_grad_kernel(GradArgs a) {
    extern __shared__ int s_live[];   // [N] live particles of the current jet, ascending
    __shared__ int s_n, s_one, s_cnt[4];
    __shared__ double s_acc[3];
    const int tid = threadIdx.x, N = a.N;
    float* base = a.ws + (size_t)blockIdx.x * a.R.floats;
    if (a.want_grad)
        for (size_t e = tid; e < 2 * a.Lo.total; e += kFp32Threads) base[a.R.slice + e] = 0.0f;
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
                for (int i = tid; i < 2 * a.f.X; i += kFp32Threads) a.d_context[((size_t)(i / a.f.X) * a.B + b) * a.f.X + i % a.f.X] = 0.0f;
            continue;
        }
        const Jet J{a.x + (size_t)b * N * a.f.Dc, a.k + (size_t)b * N, mask, a.x0 + (size_t)b * N * a.f.Dc, a.x1 + (size_t)b * N * a.f.Dc,
                    a.k1 + (size_t)b * N, b, nl, (float)nl};
        forward_jet(a, base, s_cnt, J);
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
    const Region R = make_region(make_dims(d), N, Lo.total);
    return kHeaderBytes + (size_t)grad_ctas(Lo, B) * R.floats * sizeof(float);
}

int launch_epic_loss_grad(const MmbEpicDims& d, const float* W, const float* x, const uint8_t* k, const uint8_t* mask, const float* temb,
                          int temb_stride, const float* x0, const float* x1, const uint8_t* k1, int B, int N, float* losses, float* jac,
                          float* d_context, void* workspace, cudaStream_t stream) {
    GradArgs a;
    a.W = W;
    a.Lo = mmb_epic_layout(&d);
    a.f = make_dims(d);
    a.R = make_region(a.f, N, a.Lo.total);
    a.x = x, a.k = k, a.mask = mask, a.temb = temb, a.temb_stride = temb_stride;
    a.x0 = x0, a.x1 = x1, a.k1 = k1;
    a.B = B, a.N = N, a.P = grad_ctas(a.Lo, B);
    a.part = static_cast<double*>(workspace);
    a.ws = reinterpret_cast<float*>(static_cast<char*>(workspace) + kHeaderBytes);
    a.want_grad = jac != nullptr;
    a.d_context = (jac && a.f.X) ? d_context : nullptr;
    epic_loss_grad_kernel<<<a.P, kFp32Threads, (size_t)N * sizeof(int), stream>>>(a);
    if (int rc = cuda_ok(cudaGetLastError(), "epic_loss_grad launch")) return rc;
    const size_t n_jac = jac ? 2 * a.Lo.total : 0, n_ctx = a.d_context ? (size_t)2 * B * a.f.X : 0;
    const size_t want = (n_jac + n_ctx + 255) / 256;
    const unsigned blocks = (unsigned)(want < 1 ? 1 : (want > 4096 ? 4096 : want));
    epic_grad_reduce_kernel<<<blocks, 256, 0, stream>>>(a.ws, a.R.floats, a.R.slice, a.part, a.P, n_jac, jac, a.d_context, n_ctx, losses);
    return cuda_ok(cudaGetLastError(), "epic_grad_reduce launch");
}

}  // namespace mmb
