// ggp_cell.cuh — per-cell bodies of the lineage-forest passes (host+device), FP64, strict rounding.
//
// Replaces, from the reference (paths under src/):
//   init_sc_distribution (+ _r), a cell's starting belief  predictions.h:63-82, 317-337
//   sc_likelihood (one cell of total_likelihood)           likelihood.h:36-103
//   sc_prediction_forward                                  predictions.h:93-150
//   sc_prediction_backward                                 predictions.h:368-422
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
// a cell's starting belief, on the complete 4x4 matrix (SURVEY.md H3), for every pass that walks cells: the per-thread
// bodies below, the cooperative kernels and tests/hostcheck.  mu, C out.  No __restrict__ on the helpers' arrays, and the
// root's NaN record (on_ll) stays ahead of the update: either change reschedules the strict kernels, which sit on a
// register-allocation edge (DESIGN.md 5.1b).
// ------------------------------------------------------------------------------------------------
// root (predictions.h:63-82, likelihood.h:53-69): init_cells_f sets the means and the diagonal, the off-diagonals are the
// root's persistent covariance (carry, CHAIN) or zero (carry == nullptr); then the update at the cell's first point `off`.
// on_ll receives that point's log-evidence term before the update (where the likelihood records a NaN term).
template <class OnLl>
GGP_HD void ggp_root_start(double* mu, double* C, const GgpScratch* carry, const GgpDevForest& F, const double* p, int64_t off,
                           const GgpMathTables* __restrict__ T, OnLl on_ll) {
#pragma unroll
    for (int i = 0; i < 16; ++i) C[i] = carry ? (*carry)[i] : 0.0;
    mu[0] = F.init_f[0]; mu[1] = F.init_f[1];
    C[0] = F.init_f[2];  C[5] = F.init_f[3];
    mu[2] = p[0]; mu[3] = p[3];
    C[10] = p[2] / (2. * p[1]);
    C[15] = p[5] / (2. * p[4]);
    const GgpMeas m = ggp_measure16(mu, C, F.x[off], F.g[off], p[7], p[8], F.model);
    on_ll(ggp_log_evidence(m, T));
    ggp_posterior16(mu, C, m);
}

// leaf (predictions.h:318-331): init_cells_r sets the means and the diagonal, the rest is the forward posterior at the
// cell's last point `at`; that prior goes to bwd[at] in the reversed frame, then the update at `at`.  p0 = parameters there.
GGP_HD void ggp_leaf_start(double* mu, double* C, const GgpDevForest& F, const double* fwd, double* bwd, const double* p0, int64_t at) {
    double R[16], rm[4];
    const double* fs = fwd + 20 * at;
#pragma unroll
    for (int i = 0; i < 16; ++i) C[i] = fs[4 + i];
    mu[0] = F.init_r[0]; mu[1] = F.init_r[1];
    C[0] = F.init_r[2];  C[5] = F.init_r[3];
    mu[2] = -p0[0]; mu[3] = -p0[3];
    C[10] = p0[2] / (2. * p0[1]);
    C[15] = p0[5] / (2. * p0[4]);
    ggp_reverse_mean(mu, rm);
    ggp_reverse_cov(C, R);
    ggp_store20(bwd + 20 * at, rm, R);
    const GgpMeas m = ggp_measure16(mu, C, F.x[at], F.g[at], p0[7], p0[8], F.model);
    ggp_posterior16(mu, C, m);
}

// mother (predictions.h:201-275): the final backward beliefs (bstate rows) of daughters d1, d2 (-1: none) mapped back
// through division and, with two daughters, multiplied.  p0 = the mother's parameters at her last point.
GGP_HD void ggp_mother_start(double* mu, double* C, const double* bstate, int d1, int d2, const double* p0, const GgpModel& md) {
    const double* b1 = bstate + 20 * (int64_t)(d1 >= 0 ? d1 : d2);
#pragma unroll
    for (int i = 0; i < 4; ++i) mu[i] = b1[i];
#pragma unroll
    for (int i = 0; i < 16; ++i) C[i] = b1[4 + i];
    ggp_divide_r16(mu, C, p0[9], p0[10], md);
    if (d1 >= 0 && d2 >= 0) {
        const double* b2 = bstate + 20 * (int64_t)d2;
        double mu2[4], C2[16];
#pragma unroll
        for (int i = 0; i < 4; ++i) mu2[i] = b2[i];
#pragma unroll
        for (int i = 0; i < 16; ++i) C2[i] = b2[4 + i];
        ggp_divide_r16(mu2, C2, p0[9], p0[10], md);
        ggp_multiply_gaussian(mu, C, mu2, C2);
    }
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
        const GgpScratch carry{Cc, 1};
        double mu[4], C[16];
        ggp_root_start(mu, C, CHAIN ? &carry : nullptr, F, PRED ? A.params + GGP_NP * F.seg[off] : p_lik, off, T, [&](double ll) {
            own = own + ll;
            if (!PRED && ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot]);
        });
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
        t = n - 1;
        from = off + t;
        ggp_leaf_start(mu, C, F, A.fwd, A.bwd, p0, from);
    } else {
        ggp_mother_start(mu, C, A.bstate, d1, d2, p0, F.model);
        t = n;   // virtual point: the daughters' first time
        from = F.s_off[d1 >= 0 ? d1 : d2];
    }
    ggp_state_from16(s, mu, C);
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
