// ggp_cell.cuh — per-cell bodies of the lineage-forest passes (host+device), FP64, strict rounding.
//
// Replaces, from the reference (paths under src/):
//   sc_likelihood (one cell of total_likelihood)           likelihood.h:36-103
//   sc_prediction_forward                                  predictions.h:93-150
//   sc_prediction_backward (+ init_sc_distribution_r)      predictions.h:317-337, 368-422
//   one point of combine_predictions                       predictions.h:466-499
//
// One thread runs one (cell, parameter vector) pair through these bodies.  The device passes use the
// cooperative step of ggp_coop_kernels.cuh instead (combine_predictions excepted); tests/hostcheck compiles
// the bodies for the host so whole passes can be compared bit for bit with the oracle on a machine
// without a GPU.  A cell's belief (4 means + 10 covariances) lives in
// registers for the whole cell; there is exactly ONE inlined call site of the propagation step per
// body: the division gap is treated as a virtual time step in front of the cell's first point.
#pragma once
#include <stdint.h>
#include "ggp_filter.cuh"
#include "ggp_linalg.cuh"

#if defined(__CUDA_ARCH__)
#define GGP_NAN_MIN(ptr, val) atomicMin((ptr), (unsigned long long)(val))
#else
#define GGP_NAN_MIN(ptr, val) do { if ((unsigned long long)(val) < *(ptr)) *(ptr) = (unsigned long long)(val); } while (0)
#endif

GGP_HD GgpOuParams ggp_ou(const double* __restrict__ p, bool flip) {
    GgpOuParams o;
    o.ml = flip ? -p[0] : p[0]; o.gl = p[1]; o.sl2 = p[2];
    o.mq = flip ? -p[3] : p[3]; o.gq = p[4]; o.sq2 = p[5];
    o.b = flip ? -p[6] : p[6];
    return o;
}

GGP_HD void ggp_store20(double* __restrict__ dst, const double* __restrict__ mean, const double* __restrict__ C) {
#if defined(__CUDA_ARCH__)
    double2* d = reinterpret_cast<double2*>(dst);
    d[0] = make_double2(mean[0], mean[1]);
    d[1] = make_double2(mean[2], mean[3]);
#pragma unroll
    for (int i = 0; i < 8; ++i) d[2 + i] = make_double2(C[2 * i], C[2 * i + 1]);
#else
    for (int i = 0; i < 4; ++i) dst[i] = mean[i];
    for (int i = 0; i < 16; ++i) dst[4 + i] = C[i];
#endif
}

// ------------------------------------------------------------------------------------------------
// forward filter of one cell for one parameter vector; returns the cell's own log-evidence sum.
//   PRED  = false: likelihood (likelihood.h:36-103); p_lik = the vector's 11 parameters
//   PRED  = true : prediction_forward (predictions.h:93-150); parameters per segment, posteriors stored
//   CHAIN = true : a root evaluated for successive vectors by the same thread; Cc = its persistent
//                  covariance (MOMAdata::cov), in/out, so each vector starts from the off-diagonals the
//                  previous one left (SURVEY.md H3)
// v = vector index inside the chunk.
// ------------------------------------------------------------------------------------------------
template <bool PRED, bool CHAIN>
GGP_HD double ggp_cell_forward(const GgpDevForest& F, const GgpFwdArgs& A, int slot, int v,
                               const double* __restrict__ p_lik, const GgpMathTables* __restrict__ T,
                               const GgpScratch& S, double* __restrict__ Cc) {
    const int64_t off = F.s_off[slot];
    const int n = F.s_n[slot];
    const int parent = F.s_parent[slot];
    const int64_t vstride = (int64_t)A.v_count * F.n_cells;
    const int64_t vbase = (int64_t)(PRED ? 0 : v) * F.n_cells;
    double own = 0.0;
    GgpState s;
    int t;
    int64_t from;   // ctp the next propagation starts from
    if (parent < 0) {
        // ---- root: first update on the full matrix (stale off-diagonals) ----
        const double* p = PRED ? A.params + GGP_NP * F.seg[off] : p_lik;
        double mu[4], C[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) C[i] = CHAIN ? Cc[i] : 0.0;
        mu[0] = F.init_f[0]; mu[1] = F.init_f[1];
        C[0] = F.init_f[2];  C[5] = F.init_f[3];
        mu[2] = p[0]; mu[3] = p[3];
        C[10] = p[2] / (2. * p[1]);
        C[15] = p[5] / (2. * p[4]);
        const GgpMeas m = ggp_measure16(mu, C, F.x[off], F.g[off], p[7], p[8], F.model);
        const double ll = ggp_log_evidence(m, T);
        own = own + ll;
        if (!PRED && ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot]);
        ggp_posterior16(mu, C, m);
        if (PRED) ggp_store20(A.out_fwd + 20 * off, mu, C);
        if (CHAIN) {
#pragma unroll
            for (int i = 0; i < 16; ++i) Cc[i] = C[i];
        }
        ggp_state_from16(s, mu, C);
        t = 0;
        from = off;
    } else {
        // ---- daughter: mother's last posterior; the division gap is step "-1" ----
#pragma unroll
        for (int k = 0; k < 4; ++k) s.m[k] = A.state[k * vstride + vbase + parent];
#pragma unroll
        for (int k = 0; k < 10; ++k) s.c[k] = A.state[(4 + k) * vstride + vbase + parent];
        t = -1;
        from = F.s_off[parent] + F.s_n[parent] - 1;
    }
    while (t + 1 < n) {
        const double* pp = PRED ? A.params + GGP_NP * F.seg[from] : p_lik;
        const double dt = F.time[off + t + 1] - F.time[from];
        ggp_propagate(s, dt, ggp_ou(pp, false), T, S);
        if (t < 0) ggp_divide(s, pp[9], pp[10], F.model);
        ++t;
        from = off + t;
        const double* pt = PRED ? A.params + GGP_NP * F.seg[from] : p_lik;
        const GgpMeas m = ggp_measure(s, s.c[1], F.x[from], F.g[from], pt[7], pt[8], F.model);
        const double ll = ggp_log_evidence(m, T);
        own = own + ll;
        if (!PRED && ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot] + t);
        if (PRED) {
            double C[16];
            ggp_posterior(s, s.c[1], m, C);
            ggp_store20(A.out_fwd + 20 * from, s.m, C);
        } else if (CHAIN && t == n - 1) {
            ggp_posterior(s, s.c[1], m, Cc);
        } else {
            ggp_posterior(s, s.c[1], m, nullptr);
        }
    }
    if (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) A.state[k * vstride + vbase + slot] = s.m[k];
#pragma unroll
        for (int k = 0; k < 10; ++k) A.state[(4 + k) * vstride + vbase + slot] = s.c[k];
    }
    if (!PRED && A.cell_ll) A.cell_ll[(int64_t)(A.v0 + v) * F.n_cells + F.s_cell[slot]] = own;
    return own;
}

// ------------------------------------------------------------------------------------------------
// backward filter of one cell (predictions.h:368-422), cells processed from the leaves upward
// ------------------------------------------------------------------------------------------------
GGP_HD void ggp_cell_backward(const GgpDevForest& F, const GgpBwdArgs& A, int slot, const GgpMathTables* __restrict__ T,
                              const GgpScratch& S) {
    const int64_t off = F.s_off[slot];
    const int n = F.s_n[slot];
    const int d1 = F.s_d1[slot], d2 = F.s_d2[slot];
    double mu[4], C[16], R[16], rm[4];
    GgpState s;
    int t;
    int64_t from;
    const double* p0 = A.params + GGP_NP * F.seg[off + n - 1];
    if (d1 < 0 && d2 < 0) {
        // leaf (predictions.h:318-331): means and diagonal reset, the rest is the forward posterior
        t = n - 1;
        from = off + t;
        const double* fs = A.fwd + 20 * from;
#pragma unroll
        for (int i = 0; i < 16; ++i) C[i] = fs[4 + i];
        mu[0] = F.init_r[0]; mu[1] = F.init_r[1];
        C[0] = F.init_r[2];  C[5] = F.init_r[3];
        mu[2] = -p0[0]; mu[3] = -p0[3];
        C[10] = p0[2] / (2. * p0[1]);
        C[15] = p0[5] / (2. * p0[4]);
        ggp_reverse_mean(mu, rm);
        ggp_reverse_cov(C, R);
        ggp_store20(A.bwd + 20 * from, rm, R);
        const GgpMeas m = ggp_measure16(mu, C, F.x[from], F.g[from], p0[7], p0[8], F.model);
        ggp_posterior16(mu, C, m);
        ggp_state_from16(s, mu, C);
    } else {
        // mother (predictions.h:201-275): daughters' beliefs mapped back through division and multiplied
        const int da = d1 >= 0 ? d1 : d2;
        const double* b1 = A.bstate + 20 * (int64_t)da;
#pragma unroll
        for (int i = 0; i < 4; ++i) mu[i] = b1[i];
#pragma unroll
        for (int i = 0; i < 16; ++i) C[i] = b1[4 + i];
        ggp_divide_r16(mu, C, p0[9], p0[10], F.model);
        if (d1 >= 0 && d2 >= 0) {
            const double* b2 = A.bstate + 20 * (int64_t)d2;
            double mu2[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) mu2[i] = b2[i];
#pragma unroll
            for (int i = 0; i < 16; ++i) R[i] = b2[4 + i];
            ggp_divide_r16(mu2, R, p0[9], p0[10], F.model);
            ggp_multiply_gaussian(mu, C, mu2, R);
        }
        ggp_state_from16(s, mu, C);
        t = n;   // virtual point: the daughters' first time
        from = F.s_off[da];
    }
    while (t > 0) {
        const double* pp = A.params + GGP_NP * F.seg[off + t - 1];
        const double dt = F.time[from] - F.time[off + t - 1];
        ggp_propagate(s, dt, ggp_ou(pp, true), T, S);
        --t;
        from = off + t;
        ggp_state_to16(s, C);
        ggp_reverse_mean(s.m, rm);
        ggp_reverse_cov(C, R);
        ggp_store20(A.bwd + 20 * from, rm, R);
        const GgpMeas m = ggp_measure(s, s.c[1], F.x[from], F.g[from], pp[7], pp[8], F.model);
        ggp_posterior(s, s.c[1], m, C);
#pragma unroll
        for (int i = 0; i < 4; ++i) mu[i] = s.m[i];
    }
    ggp_store20(A.bstate + 20 * (int64_t)slot, mu, C);
}

// ------------------------------------------------------------------------------------------------
// combine_predictions for one ctp (predictions.h:466-499): N(fwd) * N(bwd) / prior
// ------------------------------------------------------------------------------------------------
GGP_HD void ggp_ctp_combine(const double* __restrict__ f20, const double* __restrict__ b20, const double* __restrict__ p,
                            double* __restrict__ out20) {
    double m1[4], c1[16], m2[4], c2[16];
#pragma unroll
    for (int k = 0; k < 4; ++k) { m1[k] = f20[k]; m2[k] = b20[k]; }
#pragma unroll
    for (int k = 0; k < 16; ++k) { c1[k] = f20[4 + k]; c2[k] = b20[4 + k]; }
    ggp_multiply_gaussian(m1, c1, m2, c2);
    ggp_divide_by_prior(m1, c1, p);
    ggp_store20(out20, m1, c1);
}
