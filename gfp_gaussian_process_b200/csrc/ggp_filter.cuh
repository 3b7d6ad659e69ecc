// ggp_filter.cuh — the per-time-point measurement update, its log-evidence term and the cell-division
// maps (forward and backward) of the lineage filter, in registers.
//
// Replaces, from the reference (paths under src/):
//   posterior()                    predictions.h:84-89
//   log_likelihood()               likelihood.h:26-32
//   loop body of sc_likelihood()   likelihood.h:53-69, :95
//   mean_cov_after_division()      predictions.h:18-61     (+ mean_cov_after_division_r :201-275)
// A cell's starting belief (init_sc_distribution, predictions.h:63-82, + _r :317-337) is built from these in ggp_cell.cuh.
//
// The reference does this with heap-allocated Eigen matrices; here the belief is 4 means + the upper
// triangle (+ the one lower element a measurement can see, c10) in registers.  The Eigen expression
// semantics that fix the rounding are kept (SURVEY.md H5): the 2x2 inverse is 1/det times cofactors,
// det(S) in the log term comes from a partially pivoted LU, products are accumulated left to right.
// Host+device like the rest of the strict path; compile with FMA contraction off.
#pragma once
#include "ggp_step.cuh"

#define GGP_TWO_LOG_2PI 3.6757541328186907   /* 2*log(2*M_PI), likelihood.h:31 (same bits from libm and MPFR) */
#define GGP_LOG2 0.6931471805599453          /* log(2.), predictions.h:37,205 */


struct GgpMeas {
    double xg0, xg1;
    double Si00, Si01, Si10, Si11;
    double S00, S01, S10, S11;
};

// S = C[0:2,0:2] + D, Si = S^-1 (likelihood.h:54-67).  c10 = the (1,0) element of the covariance; it equals
// s.c[1] except at a root's / leaf's first update when stale state is carried (SURVEY.md H3).
GGP_HD GgpMeas ggp_measure(const GgpState& s, double c10, double x, double g, double var_x, double var_g,
                           const GgpModel& md) {
    GgpMeas m;
    m.xg0 = x - s.m[0];
    m.xg1 = g - s.m[1];
    double D11 = md.noise_scaled ? var_g * (s.m[1] + md.fp_auto) : var_g;
    m.S00 = s.c[0] + var_x;
    m.S01 = s.c[1] + 0.0;
    m.S10 = c10 + 0.0;
    m.S11 = s.c[4] + D11;
    double det = m.S00 * m.S11 - m.S10 * m.S01;
    double invdet = 1.0 / det;
    m.Si00 = m.S11 * invdet;
    m.Si10 = -m.S10 * invdet;
    m.Si01 = -m.S01 * invdet;
    m.Si11 = m.S00 * invdet;
    return m;
}

// -1/2 r^T Si r - 1/2 log det S - 2 log 2pi (likelihood.h:26-32; the constant is as written there), in two pieces so that
// the cooperative likelihood step can evaluate the second one (a serial chain: division, log) off its critical path.
GGP_HD double ggp_log_evidence_quad(const GgpMeas& m) {
    double r0 = (-0.5 * m.xg0) * m.Si00 + (-0.5 * m.xg1) * m.Si10;
    double r1 = (-0.5 * m.xg0) * m.Si01 + (-0.5 * m.xg1) * m.Si11;
    return r0 * m.xg0 + r1 * m.xg1;
}
GGP_HD double ggp_log_evidence_finish(double a, double S00, double S01, double S10, double S11, const GgpMathTables* __restrict__ M) {
    // determinant of the dynamic-size copy: partial-pivot LU
    double p00 = S00, p01 = S01, p10 = S10, p11 = S11, sign = 1.0;
    if (fabs(p10) > fabs(p00)) {
        double t0 = p00, t1 = p01;
        p00 = p10; p01 = p11; p10 = t0; p11 = t1;
        sign = -1.0;
    }
    if (p00 != 0.0) p10 = p10 / p00;
    p11 = p11 - p10 * p01;
    double det = sign * (p00 * p11);
    return a - 0.5 * ggp_log(det, M) - GGP_TWO_LOG_2PI;
}
GGP_HD double ggp_log_evidence(const GgpMeas& m, const GgpMathTables* __restrict__ M) {
    return ggp_log_evidence_finish(ggp_log_evidence_quad(m), m.S00, m.S01, m.S10, m.S11, M);
}

// Kalman update of mean and upper triangle (predictions.h:84-89).  If full16 != nullptr the complete
// row-major 4x4 posterior covariance (whose two triangles differ in the last bits, because the reference
// evaluates K^T Si K entry by entry) is written there as well.
GGP_HD void ggp_posterior(GgpState& s, double c10, const GgpMeas& m, double* __restrict__ full16) {
    // K = C[0:2, :]; T = K^T Si
    const double K0[4] = {s.c[0], s.c[1], s.c[2], s.c[3]};
    const double K1[4] = {c10, s.c[4], s.c[5], s.c[6]};
    double T0[4], T1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        T0[i] = K0[i] * m.Si00 + K1[i] * m.Si10;
        T1[i] = K0[i] * m.Si01 + K1[i] * m.Si11;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) s.m[i] = s.m[i] + ((0.0 + T0[i] * m.xg0) + T1[i] * m.xg1);
    if (full16) {
        // symmetric prior except (0,1)/(1,0): element (i,j) of the prior
        const double C[16] = {s.c[0], s.c[1], s.c[2], s.c[3], c10, s.c[4], s.c[5], s.c[6],
                              s.c[2], s.c[5], s.c[7], s.c[8], s.c[3], s.c[6], s.c[8], s.c[9]};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) full16[4 * i + j] = C[4 * i + j] - (T0[i] * K0[j] + T1[i] * K1[j]);
    }
    double n[10];
    n[0] = s.c[0] - (T0[0] * K0[0] + T1[0] * K1[0]);
    n[1] = s.c[1] - (T0[0] * K0[1] + T1[0] * K1[1]);
    n[2] = s.c[2] - (T0[0] * K0[2] + T1[0] * K1[2]);
    n[3] = s.c[3] - (T0[0] * K0[3] + T1[0] * K1[3]);
    n[4] = s.c[4] - (T0[1] * K0[1] + T1[1] * K1[1]);
    n[5] = s.c[5] - (T0[1] * K0[2] + T1[1] * K1[2]);
    n[6] = s.c[6] - (T0[1] * K0[3] + T1[1] * K1[3]);
    n[7] = s.c[7] - (T0[2] * K0[2] + T1[2] * K1[2]);
    n[8] = s.c[8] - (T0[2] * K0[3] + T1[2] * K1[3]);
    n[9] = s.c[9] - (T0[3] * K0[3] + T1[3] * K1[3]);
#pragma unroll
    for (int i = 0; i < 10; ++i) s.c[i] = n[i];
}

// mother's last posterior -> daughter's prior (predictions.h:18-61); s already propagated over the gap
GGP_HD void ggp_divide(GgpState& s, double var_dx, double var_dg, const GgpModel& md) {
    if (md.division_binomial) {
        double c00 = s.c[0] + var_dx;
        double c01 = s.m[1] / 2. * var_dx + s.c[1];
        double c11 = var_dx * (s.m[1] * s.m[1] + s.c[4]) / 2. + var_dg * s.m[1] / 4. * (1 - var_dx) + s.c[4] / 4.;
        s.c[0] = c00; s.c[1] = c01; s.c[4] = c11;
        s.c[5] = s.c[5] / 2;
        s.c[6] = s.c[6] / 2;
    } else {   // D + F C F^T, F = diag(1, 1/2, 1, 1)
        s.c[0] = var_dx + s.c[0];
        s.c[1] = 0.0 + (s.c[1] * 0.5);
        s.c[4] = var_dg + (0.5 * s.c[4]) * 0.5;
        s.c[5] = 0.0 + (0.5 * s.c[5]);
        s.c[6] = 0.0 + (0.5 * s.c[6]);
        s.c[2] = 0.0 + s.c[2]; s.c[3] = 0.0 + s.c[3]; s.c[7] = 0.0 + s.c[7]; s.c[8] = 0.0 + s.c[8]; s.c[9] = 0.0 + s.c[9];
    }
    s.m[0] = s.m[0] + -GGP_LOG2;
    s.m[1] = 0.5 * s.m[1] + 0.0;
}

// ---- full-matrix variants -----------------------------------------------------------------------
// The reference keeps a full 4x4 MOMAdata::cov whose two triangles need not agree: posterior() fills
// every entry separately, and a root (forward) or leaf (backward) starts from whatever an earlier pass
// left off the diagonal (SURVEY.md H3).  These variants work on the complete row-major matrix; they
// are used once per cell (first update of a root/leaf), the register version above everywhere else.
GGP_HD GgpMeas ggp_measure16(const double* __restrict__ mean, const double* __restrict__ C, double x, double g,
                             double var_x, double var_g, const GgpModel& md) {
    GgpState s;
    s.m[0] = mean[0]; s.m[1] = mean[1];
    s.c[0] = C[0]; s.c[1] = C[1]; s.c[4] = C[5];
    return ggp_measure(s, C[4], x, g, var_x, var_g, md);
}

GGP_HD void ggp_posterior16(double* __restrict__ mean, double* __restrict__ C, const GgpMeas& m) {
    double T0[4], T1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        T0[i] = C[i] * m.Si00 + C[4 + i] * m.Si10;
        T1[i] = C[i] * m.Si01 + C[4 + i] * m.Si11;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) mean[i] = mean[i] + ((0.0 + T0[i] * m.xg0) + T1[i] * m.xg1);
    double n[16];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) n[4 * i + j] = C[4 * i + j] - (T0[i] * C[j] + T1[i] * C[4 + j]);
#pragma unroll
    for (int i = 0; i < 16; ++i) C[i] = n[i];
}

GGP_HD void ggp_state_from16(GgpState& s, const double* __restrict__ mean, const double* __restrict__ C) {
    s.m[0] = mean[0]; s.m[1] = mean[1]; s.m[2] = mean[2]; s.m[3] = mean[3];
    s.c[0] = C[0]; s.c[1] = C[1]; s.c[2] = C[2]; s.c[3] = C[3]; s.c[4] = C[5];
    s.c[5] = C[6]; s.c[6] = C[7]; s.c[7] = C[10]; s.c[8] = C[11]; s.c[9] = C[15];
}

GGP_HD void ggp_state_to16(const GgpState& s, double* __restrict__ C) {   // symmetric expansion
    C[0] = s.c[0]; C[1] = s.c[1]; C[2] = s.c[2]; C[3] = s.c[3];
    C[4] = s.c[1]; C[5] = s.c[4]; C[6] = s.c[5]; C[7] = s.c[6];
    C[8] = s.c[2]; C[9] = s.c[5]; C[10] = s.c[7]; C[11] = s.c[8];
    C[12] = s.c[3]; C[13] = s.c[6]; C[14] = s.c[8]; C[15] = s.c[9];
}

// one daughter's belief at its first point mapped back through division (predictions.h:213-238 / :243-266);
// mean/C are the daughter's final backward state (full matrix), overwritten with the mother's frame
GGP_HD void ggp_divide_r16(double* __restrict__ mean, double* __restrict__ C, double var_dx, double var_dg,
                           const GgpModel& md) {
    if (md.division_binomial) {
        C[0] = C[0] + var_dx;
        C[5] = 8. * var_dx * (mean[1] * mean[1] + C[5]) + 2. * var_dg * mean[1] + 8. * C[5];
        double c01 = 2. * mean[1] * var_dx + 4. * C[1];
        C[1] = c01; C[4] = c01;
        C[9] = C[9] * 2; C[6] = C[6] * 2;
        C[13] = C[13] * 2; C[7] = C[7] * 2;
        mean[0] = mean[0] + GGP_LOG2;
        mean[1] = mean[1] * 2;
    } else {   // D + F C F^T, F = diag(1, 2, 1, 1)
        mean[0] = mean[0] + GGP_LOG2;
        mean[1] = 2 * mean[1] + 0.0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double fi = (i == 1) ? 2.0 : 1.0, fj = (j == 1) ? 2.0 : 1.0;
                const double d = (i == j) ? (i == 0 ? var_dx : (i == 1 ? var_dg : 0.0)) : 0.0;
                C[4 * i + j] = d + (fi * C[4 * i + j]) * fj;
            }
    }
}
