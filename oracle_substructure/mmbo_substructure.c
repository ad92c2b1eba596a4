/*
 * mmbo_substructure.c — CPU restatement of mmb_jet_substructure: N-subjettiness tau1..tau3 on exclusive kt / WTA_pt axes and
 * the energy correlation functions e2, e3, D2 (the observables of JetClassHighLevelFeatures.substructure,
 * mp/data/particle_clouds/jets.py:204-240).  TEST INFRASTRUCTURE ONLY (see mmbo_substructure.h).
 *
 * Deliberately plain: the clustering is a brute-force scan of every pair and beam distance at every step, in the
 * (lower, upper) index order of the tie rule, where the kernel keeps nearest-neighbour bookkeeping.  The two share only
 * the definitions (DESIGN.md §4.6) and the order of the fp64 operations inside one distance.
 */
#include "mmbo_substructure.h"

#include <math.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define SUB_PI 3.141592653589793
#define SUB_TWO_PI 6.283185307179586

/* dR^2 between two directions; dphi wrapped into [-pi, pi] */
static double delta_r2(double eta_a, double phi_a, double eta_b, double phi_b) {
    const double deta = eta_a - eta_b;
    double dphi = phi_a - phi_b;
    if (dphi > SUB_PI) dphi = dphi - SUB_TWO_PI;
    else if (dphi < -SUB_PI) dphi = dphi + SUB_TWO_PI;
    return deta * deta + dphi * dphi;
}

/* dR^beta from dR^2 */
static double angle_pow(double dr2, double beta) { return beta == 1.0 ? sqrt(dr2) : pow(dr2, 0.5 * beta); }

typedef struct {
    double *pt, *eta, *phi;   /* used particles, compacted in slot order */
    double *opt;              /* current pt of each clustering object */
    int *slot, *dir, *alive;  /* slot of each used particle; particle whose direction an object carries; object still present */
    double *ang;              /* [n][n] dR^beta between used particles */
} Scratch;

static void one_jet(const float* x, const uint8_t* mask, const float* mean, const float* sd, int N, float R, float beta, Scratch* s,
                    float* out, int16_t* axes) {
    for (int c = 0; c < MMB_SUB_OBS; ++c) out[c] = NAN;
    if (axes) for (int a = 0; a < 6; ++a) axes[a] = -1;

    /* inputs: (x * std + mean) in fp32, as mmb_jet_observables; used iff mask != 0 && pt > 0 */
    int n = 0;
    for (int slot = 0; slot < N; ++slot) {
        if (!mask[slot]) continue;
        float c[3];
        for (int i = 0; i < 3; ++i) c[i] = x[slot * 3 + i] * (sd ? sd[i] : 1.0f) + (mean ? mean[i] : 0.0f);
        if (!(c[0] > 0.0f)) continue;
        s->pt[n] = c[0]; s->eta[n] = c[1]; s->phi[n] = c[2]; s->slot[n] = slot;
        ++n;
    }
    if (n < 3) return;   /* undefined: NaN, axes -1 */

    /* exclusive kt clustering, WTA_pt recombination.  Candidates are visited in ascending (lower, upper) order with the beam
     * candidate of i counted as (i, i), so a strict '<' keeps the first of equal distances: the tie rule. */
    const double R2 = (double)R * (double)R, invR2 = 1.0 / R2;   /* d_ij multiplies by 1/R^2, as fastjet does */
    for (int i = 0; i < n; ++i) { s->opt[i] = s->pt[i]; s->dir[i] = i; s->alive[i] = 1; }
    int ax[6];                     /* tau1 axis | tau2 axes | tau3 axes, as indices of used particles */
    int left = n;
    for (;;) {
        if (left <= 3) {           /* the exclusive `left`-jet axes: present objects in ascending index */
            int* dst = ax + (left == 1 ? 0 : left == 2 ? 1 : 3), m = 0;
            for (int i = 0; i < n; ++i)
                if (s->alive[i]) dst[m++] = s->dir[i];
        }
        if (left == 1) break;
        double best = INFINITY;
        int lo = -1, hi = -1;
        for (int i = 0; i < n; ++i) {
            if (!s->alive[i]) continue;
            const double pti2 = s->opt[i] * s->opt[i];
            if (pti2 < best) { best = pti2; lo = i; hi = i; }           /* d_iB = pt_i^2 */
            for (int j = i + 1; j < n; ++j) {
                if (!s->alive[j]) continue;
                const double ptj2 = s->opt[j] * s->opt[j];
                const double m = pti2 < ptj2 ? pti2 : ptj2;
                const int a = s->dir[i], b = s->dir[j];
                const double d = m * delta_r2(s->eta[a], s->phi[a], s->eta[b], s->phi[b]) * invR2;   /* d_ij */
                if (d < best) { best = d; lo = i; hi = j; }
            }
        }
        if (lo == hi) {
            s->alive[lo] = 0;      /* beam step: the object leaves the sequence */
        } else {                   /* merge into the lower index; direction of the harder object, the lower index on a tie */
            if (s->opt[hi] > s->opt[lo]) s->dir[lo] = s->dir[hi];
            s->opt[lo] = s->opt[lo] + s->opt[hi];
            s->alive[hi] = 0;
        }
        --left;
    }

    /* N-subjettiness: tau_N = sum_i pt_i min_a dR(i,a)^beta / (sum_i pt_i R^beta) */
    double ptsum = 0.0;
    for (int i = 0; i < n; ++i) ptsum += s->pt[i];
    const double d0 = ptsum * angle_pow(R2, beta);
    double tau[3];
    for (int t = 0; t < 3; ++t) {
        const int* a = ax + (t == 0 ? 0 : t == 1 ? 1 : 3);
        double acc = 0.0;
        for (int i = 0; i < n; ++i) {
            double m = INFINITY;
            for (int q = 0; q <= t; ++q) {
                const double dr2 = delta_r2(s->eta[i], s->phi[i], s->eta[a[q]], s->phi[a[q]]);
                if (dr2 < m) m = dr2;
            }
            acc += s->pt[i] * angle_pow(m, beta);
        }
        tau[t] = acc / d0;
    }

    /* energy correlation functions (arXiv:1409.6298), z_i = pt_i / sum_j pt_j */
    for (int i = 0; i < n; ++i)
        for (int j = i + 1; j < n; ++j) s->ang[i * n + j] = angle_pow(delta_r2(s->eta[i], s->phi[i], s->eta[j], s->phi[j]), beta);
    double e2 = 0.0, e3 = 0.0;
    for (int i = 0; i < n; ++i) {
        const double zi = s->pt[i] / ptsum;
        for (int j = i + 1; j < n; ++j) {
            const double zj = s->pt[j] / ptsum, aij = s->ang[i * n + j];
            e2 += zi * zj * aij;
            for (int k = j + 1; k < n; ++k) e3 += zi * zj * (s->pt[k] / ptsum) * (aij * s->ang[i * n + k] * s->ang[j * n + k]);
        }
    }

    out[MMB_SUB_TAU1] = (float)tau[0]; out[MMB_SUB_TAU2] = (float)tau[1]; out[MMB_SUB_TAU3] = (float)tau[2];
    out[MMB_SUB_TAU21] = (float)(tau[1] / tau[0]); out[MMB_SUB_TAU32] = (float)(tau[2] / tau[1]);
    out[MMB_SUB_E2] = (float)e2; out[MMB_SUB_E3] = (float)e3; out[MMB_SUB_D2] = (float)(e3 / (e2 * e2 * e2));
    if (axes) for (int a = 0; a < 6; ++a) axes[a] = (int16_t)s->slot[ax[a]];
}

void mmbo_jet_substructure(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N, float R, float beta,
                           float* out, int16_t* axes) {
#pragma omp parallel
    {
        Scratch s;
        const size_t n = N > 0 ? (size_t)N : 1;
        double* d = malloc(sizeof(double) * (4 * n + n * n));
        int* k = malloc(sizeof(int) * 3 * n);
        s.pt = d; s.eta = d + n; s.phi = d + 2 * n; s.opt = d + 3 * n; s.ang = d + 4 * n;
        s.slot = k; s.dir = k + n; s.alive = k + 2 * n;
#pragma omp for schedule(dynamic, 16)
        for (int b = 0; b < B; ++b)
            one_jet(x + (size_t)b * N * 3, mask + (size_t)b * N, mean, sd, N, R, beta, &s, out + (size_t)b * MMB_SUB_OBS,
                    axes ? axes + (size_t)b * 6 : NULL);
        free(d);
        free(k);
    }
}

int mmbo_substructure_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
