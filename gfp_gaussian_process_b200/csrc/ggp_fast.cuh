// ggp_fast.cuh — the FAST likelihood step: same model and same moments as mean_cov_model() (reference
// src/mean_cov_model.h:73-274), different evaluation, NOT bit-identical to the reference.  Log-likelihood only
// (-m, -s, BASELINE configs[1] and [3]); predictions and joints stay on the strict path.
//
// Why it exists (SURVEY.md H1, H2): the strict path reproduces the reference's rounding bit for bit, which costs
// 66 exp + 14 Dawson + 3 pow per step, forbids FMA, and keeps the reference's ill-conditioning (integrals formed as
// differences of exp * Dawson products divided by a^(k+1/2), a = C_ll / 2 ~ 3e-7; covariances as raw second moments minus
// squared means).  Here:
//   * the integrals  I_k(B, c; t0, t1) = int s^k exp(a s^2 + B s + c) ds  are evaluated by Gauss-Legendre quadrature.  The
//     integrand is entire and nearly linear in the exponent over one time step (|a t^2 + B t| ~ 1e-2 on real data), so N
//     nodes integrate it to rounding error; every term of the sum is positive: no cancellation, no Dawson function, no
//     division by powers of a.  All 39 integrals of a step share 3 N exponentials: exp(a s^2 + B0 s), exp(a s^2 + W s) on
//     [0, t] and exp(a s'^2 + W s') on [t, 2t]; the -gq / +gq variants and the nine constants c only multiply these by
//     factors that depend on the parameters and dt alone (cached while dt repeats).  A step forms 12 quadrature sums: the six
//     moments of the B-family (exp(a s^2 + B0 s)) that the means and the g-row use, and six sums of the W-family, one per
//     state monomial of E[production^2], the one expression that reads the W-family (GgpFastNode).
//   * the g-row of the new covariance is written in CENTRAL form.  With  G1 = mq J_B[0] + dq J_Bm[0] + Clq J_Bm[1]
//     (the production integral: mean_g = bg e^{-b t} + G1), G2 the same with one more power of s, dq = bq + Cxq - mq:
//         cov(g, y) = e^{-gamma_y t} (e^{-b t} C_gy + C_xy G1 + C_ly G2 + C_qy J_Bm[0] [+ OU noise term for y = q])
//     for y = lambda, q, and the analogous x row; cov_gg = C_gg e^{-2bt} + 2 e^{-bt} (C_xg G1 + C_gl G2 + C_gq J_Bm[0])
//     + S2 - G1^2.  These are the reference's formulas (mean_cov_model.h:97-192) with the "- nm(1) * nm(i)" products expanded
//     and cancelled analytically; algebraically identical, far better conditioned.
//   * FMA contraction is allowed (this header is compiled with -fmad=true), exp / log are the CUDA library's.
// Accuracy: differs from the reference by the reference's own rounding noise (tools/ulp_envelope.py measures that
// envelope); the gate is |dloglik| / |loglik| <= 1e-10 against the oracle (tests/test_gpu_fast.py), and
// tests/hostcheck/fastcheck.cpp compares both with a binary128 evaluation.
// Validity: the quadrature order N is fixed at compile time; a step whose exponent varies by more than GGP_FAST_LMAX over
// the step (or whose C_ll is negative / not finite) raises the evaluation's `invalid` flag and the caller re-runs that
// parameter vector on the strict path.
//
// Templated on the scalar type so that the same code runs in binary128 on the host (the "truth" of the gate report).
#pragma once
#include "ggp_types.cuh"
#include "ggp_gl_tables.h"

#ifndef GGP_FAST_N
#define GGP_FAST_N 6
#endif

template <class T> struct GgpFx;   // scalar helpers

// Taylor coefficients 1/k!, k = 15 .. 2, of the short exponentials below.  On the device they live in the constant bank: an
// FP64 instruction reads such an operand as c[bank][offset], whereas a 64-bit literal costs two move instructions every time
// it is materialised (the CUDA library's exp inlined once per quadrature node: 308 of the kernel's 2 712 instructions were
// such moves, 15 % of the executed instructions; profiles/r02_fast5_gen5.txt).
#define GGP_FEXP_INIT {0x1.ae7f3e733b81fp-41, 0x1.93974a8c07c9dp-37, 0x1.6124613a86d09p-33, 0x1.1eed8eff8d898p-29, 0x1.ae64567f544e4p-26, \
                       0x1.27e4fb7789f5cp-22, 0x1.71de3a556c734p-19, 0x1.a01a01a01a01ap-16, 0x1.a01a01a01a01ap-13, 0x1.6c16c16c16c17p-10, \
                       0x1.1111111111111p-7, 0x1.5555555555555p-5, 0x1.5555555555555p-3, 0.5}
#define GGP_FEXP_MAXDEG 15
#if defined(__CUDACC__)
__constant__ double ggp_fexp_c[14] = GGP_FEXP_INIT;
#endif
GGP_HDM double ggp_fexp_k(int i) {   // 1 / (GGP_FEXP_MAXDEG - i)!
#if defined(__CUDA_ARCH__)
    return ggp_fexp_c[i];
#else
    constexpr double v[14] = GGP_FEXP_INIT;
    return v[i];
#endif
}

template <> struct GgpFx<double> {
    static GGP_HDM double exp_(double x) { return exp(x); }
    static GGP_HDM double log_(double x) { return log(x); }
    static GGP_HDM double expm1_(double x) { return expm1(x); }
    static GGP_HDM double abs_(double x) { return fabs(x); }
    static GGP_HDM bool finite_(double x) { return x - x == 0.0; }
    static GGP_HDM double ln2() { return 0.6931471805599453; }
    // Taylor polynomial of exp of degree DEG (4 .. 15), Horner; relative truncation error |x|^(DEG+1) / (DEG+1)!
    template <int DEG>
    static GGP_HDM double exp_taylor_(double x) {
        double p = ggp_fexp_k(GGP_FEXP_MAXDEG - DEG);
#pragma unroll
        for (int i = GGP_FEXP_MAXDEG - DEG + 1; i < 14; ++i) p = p * x + ggp_fexp_k(i);
        p = p * x + 1.0;
        return p * x + 1.0;
    }
    static GGP_HDM double exp_mid_(double x) { return exp_taylor_<15>(x); }     // |x| <= 0.5: 7e-19
    static GGP_HDM double exp_small_(double x) { return exp_taylor_<10>(x); }   // |x| <= 0.125: 3e-18
    static GGP_HDM double exp_small8_(double x) { return exp_taylor_<8>(x); }   // |x| <= 0.06: 3e-17
    static GGP_HDM double exp_tiny_(double x) { return exp_taylor_<6>(x); }     // |x| <= 0.01: 2e-18
    static GGP_HDM double exp_tiny4_(double x) { return exp_taylor_<4>(x); }    // |x| <= 0.001: 8e-18
};
// ranges of exp_mid_ / exp_small_ / exp_small8_ / exp_tiny_ / exp_tiny4_
#define GGP_FAST_MID 0.5
#define GGP_FAST_SMALL 0.125
#define GGP_FAST_SMALL8 0.06
#define GGP_FAST_TINY 0.01
#define GGP_FAST_TINY4 0.001

// largest |d(exponent)/ds| * t a step may have for the N-node rule to integrate s^k exp(lambda s), k = 0..3, over [0, t] and
// [t, 2t] to 3e-15 relative (measured against mpmath)
template <int N> struct GgpFastLmax;
template <> struct GgpFastLmax<3> { static GGP_HDM constexpr double v() { return 0.004; } };
template <> struct GgpFastLmax<4> { static GGP_HDM constexpr double v() { return 0.02; } };
template <> struct GgpFastLmax<5> { static GGP_HDM constexpr double v() { return 0.12; } };
template <> struct GgpFastLmax<6> { static GGP_HDM constexpr double v() { return 0.5; } };
template <> struct GgpFastLmax<8> { static GGP_HDM constexpr double v() { return 1.8; } };
template <> struct GgpFastLmax<10> { static GGP_HDM constexpr double v() { return 4.0; } };
template <> struct GgpFastLmax<12> { static GGP_HDM constexpr double v() { return 6.0; } };
template <> struct GgpFastLmax<16> { static GGP_HDM constexpr double v() { return 10.0; } };

// the N-node rule as an object (host checks pass a binary128 rule instead)
template <int N>
struct GgpGLRule {
    GGP_HDM double xi(int j) const { return GgpGL<N>::xi(j); }
    GGP_HDM double om(int j) const { return GgpGL<N>::om(j); }
};

template <class T>
struct GgpFastState {
    T m[4];    // mean: x, g, lambda, q
    T c[10];   // covariance, upper triangle row-major: xx xg xl xq gg gl gq ll lq qq
};

// what depends on the parameters and dt only (tabulated per distinct dt on the device, recomputed on change on the host).
// Everything the quadrature sums need is pre-multiplied here, so that a step spends one FMA per (node, moment).
//
// E[production^2] (S2 in ggp_fast_propagate) is a linear form in the W-family sums whose coefficients depend on the state only
// through the six monomials  1, Clq, e2, e2^2 + Cqq, Clq e2, Clq^2  (e2 = bq + 2 Cxq - mq).  So the node weights of the
// W-family are summed per MONOMIAL: Z_m = sum_j (al[m]_j exp(a s^2 + W s) + be[m]_j exp(a s'^2 + W s')), s' = t + s, and
// S2 = exp(c5) sum_m mono_m Z_m.  With R = exp(-gq s), Rh = exp(-gq s'), u = t - s, hs = sq2 / (2 gq), cq = 2 mq / gq:
//   m   al[m]                                            be[m]
//   0   mq^2 w s - hs w s R - (hs / gq) w expm1(-gq s)  mq^2 w u - hs w u Rh - (hs / gq) w expm1(-gq u)
//   1   -cq w s expm1(-gq s)                             -cq w s' R expm1(-gq u)
//   2   -cq w expm1(-gq s)                               -cq w R expm1(-gq u)
//   3   w s R                                            w u Rh
//   4   2 w s^2 R                                        2 w s' u Rh
//   5   w s^3 R                                          w s'^2 u Rh
// (mean_cov_model.h:124-164 with the moments of [0, t] and [t, 2t] collected per monomial; the differences of nearly equal
// exponentials that the collection produces - 1 - R, R - exp(-gq t), 1 - exp(-gq u) - are formed with expm1.)
template <class T>
struct alignas(16) GgpFastNode {  // one quadrature node, 20 values = 160 bytes: read with 128-bit loads
    T s, s2;                      // s_j = t xi_j and its square (exponent arguments)
    T w, ws;                      // weight w_j = t om_j, w_j s_j
    T wR, wRs, wRs2;              // w_j exp(-gq s_j) s_j^k
    T wSh;                        // w_j (exp(+gq s_j) - exp(-gq s_j))
    T al[6], be[6];               // weights of Z_m on [0, t] and [t, 2t] (table above)
};
template <class T, int N>
struct alignas(16) GgpFastConsts {
    T t;                          // the dt these were computed for
    T ebt, egl, egq;              // exp(-b t), exp(-gl t), exp(-gq t)
    T oi;                         // (1 - exp(-gl t)) / gl
    T kxx, kxl, kll, kqq;         // OU noise contributions to cov_xx, cov_xl, cov_ll, cov_qq
    T hsq;                        // sq2 / (2 gq)
    GgpFastNode<T> node[N];
};

// the constants of one step without the nodes
template <class T, int N>
GGP_HD void ggp_fast_consts_head(GgpFastConsts<T, N>& K, T t, T gl, T sl2, T gq, T sq2, T b) {
    typedef GgpFx<T> X;
    K.t = t;
    K.ebt = X::exp_(-b * t);
    K.egl = X::exp_(-gl * t);
    K.egq = X::exp_(-gq * t);
    const T igl = T(1) / gl;
    const T igq = T(1) / gq;
    const T omegl = -X::expm1_(-gl * t);
    K.oi = omegl * igl;
    // mean_cov_model.h:93-95, 117-119, 196-208: the terms without state
    K.kxx = sl2 * T(0.5) * igl * igl * igl * (T(2) * gl * t + T(4) * X::expm1_(-gl * t) - X::expm1_(T(-2) * gl * t));
    K.kxl = sl2 * T(0.5) * K.oi * K.oi;
    K.kll = sl2 * T(0.5) * igl * (-X::expm1_(T(-2) * gl * t));
    K.kqq = sq2 * T(0.5) * igq * (-X::expm1_(T(-2) * gq * t));
    K.hsq = sq2 * T(0.5) * igq;
}

// node j of a step's constants (the device gives every node a thread of its own)
template <class T, class GL>
GGP_HD void ggp_fast_consts_node(GgpFastNode<T>& n, int j, T t, T mq, T gq, T sq2, const GL& gln) {
    typedef GgpFx<T> X;
    const T igq = T(1) / gq;
    const T hs = sq2 * T(0.5) * igq, hs2 = hs * igq, mq2 = mq * mq, cq = T(2) * mq * igq;
    const T s = t * gln.xi(j), w = t * gln.om(j), sh = t + s, u = t * (1.0 - gln.xi(j));
    const T R = X::exp_(-gq * s), Rp = X::exp_(gq * s);
    const T Em = X::expm1_(-gq * s), Eu = X::expm1_(-gq * u);   // R - 1, exp(-gq (t - s)) - 1
    n.s = s; n.s2 = s * s;
    n.w = w; n.ws = w * s;
    const T wR = w * R;
    n.wR = wR; n.wRs = wR * s; n.wRs2 = wR * (s * s);
    n.wSh = w * (Rp - R);
    const T wRh = wR * X::exp_(-gq * t), wRhu = wRh * u;
    n.al[0] = mq2 * (w * s) - hs * (wR * s) - hs2 * (w * Em);
    n.be[0] = mq2 * (w * u) - hs * wRhu - hs2 * (w * Eu);
    n.al[1] = -cq * (w * s) * Em;
    n.be[1] = -cq * (wR * sh) * Eu;
    n.al[2] = -cq * w * Em;
    n.be[2] = -cq * wR * Eu;
    n.al[3] = wR * s;
    n.be[3] = wRhu;
    n.al[4] = T(2) * wR * (s * s);
    n.be[4] = T(2) * wRhu * sh;
    n.al[5] = wR * (s * s * s);
    n.be[5] = wRhu * (sh * sh);
}

template <class T, int N, class GL>
GGP_HD void ggp_fast_consts(GgpFastConsts<T, N>& K, T t, T ml, T gl, T sl2, T mq, T gq, T sq2, T b, const GL& gln) {
    (void)ml;
    ggp_fast_consts_head(K, t, gl, sl2, gq, sq2, b);
    for (int j = 0; j < N; ++j) ggp_fast_consts_node(K.node[j], j, t, mq, gq, sq2, gln);
}

// the quadrature sums of one step.  LEVEL says which exponentials the main exponent (a s^2 + B0 s) and the two secondary ones
// (Cxl s, 2 a t s) get over this step:  3: both tiny - main below 0.06, secondary below 0.001: Taylor degrees 8 and 4 (configs[1],
// real data: growth rates of 1e-2 per minute, steps of minutes);  2: below 0.125 and 0.01: degrees 10 and 6;  1: below 0.5 and
// 0.06: degrees 15 and 8 (steps of a quarter of an hour: configs[2], what a 6-node rule accepts);  0: the library's exp.
// Every sum is one FMA per node against a pre-multiplied constant.  M[0..5]: the B-family, M[6 + m]: Z_m (GgpFastNode).
template <class T, int N, int LEVEL>
GGP_HD void ggp_fast_moments(const GgpFastConsts<T, N>& K, T a, T B0, T Cxl, T EH, T* __restrict__ M) {
    typedef GgpFx<T> X;
    const T t = K.t, twoat = T(2) * a * t;
    T MB0 = 0, MB1 = 0, MBm0 = 0, MBm1 = 0, MBm2 = 0, MBs0 = 0;
    T Z[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const GgpFastNode<T> n = K.node[j];
        const T s = n.s;
        const T xa = a * n.s2 + B0 * s, xv = Cxl * s, xu = twoat * s;
        const T A = LEVEL == 3 ? X::exp_small8_(xa) : LEVEL == 2 ? X::exp_small_(xa) : LEVEL == 1 ? X::exp_mid_(xa) : X::exp_(xa);   // exp(a s^2 + B0 s)
        const T V = LEVEL == 3 ? X::exp_tiny4_(xv) : LEVEL == 2 ? X::exp_tiny_(xv) : LEVEL == 1 ? X::exp_small8_(xv) : X::exp_(xv);
        const T U = LEVEL == 3 ? X::exp_tiny4_(xu) : LEVEL == 2 ? X::exp_tiny_(xu) : LEVEL == 1 ? X::exp_small8_(xu) : X::exp_(xu);
        const T AW = A * V;                                    // exp(a s^2 + W s), W = B0 + Cxl
        const T H = AW * (U * EH);                             // exp(a s'^2 + W s'), s' = t + s, EH = exp(t (W + a t))
        MB0 += n.w * A; MB1 += n.ws * A;
        MBm0 += n.wR * A; MBm1 += n.wRs * A; MBm2 += n.wRs2 * A;
        MBs0 += n.wSh * A;
#pragma unroll
        for (int m = 0; m < 6; ++m) {
            Z[m] += n.al[m] * AW;
            Z[m] += n.be[m] * H;
        }
    }
    M[0] = MB0; M[1] = MB1; M[2] = MBm0; M[3] = MBm1; M[4] = MBm2; M[5] = MBs0;
#pragma unroll
    for (int m = 0; m < 6; ++m) M[6 + m] = Z[m];
}

// one propagation step over K.t; returns false if the step is outside the quadrature's validity range
template <class T, int N>
GGP_HD bool ggp_fast_propagate(GgpFastState<T>& st, const GgpFastConsts<T, N>& K, T ml, T gl, T mq, T gq, T sq2, T b, T lmax) {
    typedef GgpFx<T> X;
    (void)gl; (void)sq2;
    const T bx = st.m[0], bg = st.m[1], bl = st.m[2], bq = st.m[3];
    const T Cxx = st.c[0], Cxg = st.c[1], Cxl = st.c[2], Cxq = st.c[3], Cgg = st.c[4], Cgl = st.c[5], Cgq = st.c[6],
            Cll = st.c[7], Clq = st.c[8], Cqq = st.c[9];
    const T t = K.t;
    const T a = T(0.5) * Cll;
    const T B0 = b + bl + Cxl, W = B0 + Cxl;
    // validity of the rule: the exponent a s^2 + B s, B in {B0, W} -+ gq, over [0, 2t]
    const T lam = (X::abs_(B0) > X::abs_(W) ? X::abs_(B0) : X::abs_(W)) + X::abs_(gq) + T(4) * X::abs_(a) * t;
    const bool ok = (a >= T(0)) && X::finite_(lam) && (lam * t <= lmax);

    // ---- the 12 sums of the step: sum_j (weight) * (exponential), mean_cov_model.h:9-67 by quadrature ----
    // lam t bounds |a s^2 + B s| on [0, t] and |t (W + a t)|: below GGP_FAST_SMALL (every step a rule of at most 5 nodes accepts)
    // these exponentials are short polynomials as well
    const T sec = X::abs_(Cxl) > T(2) * a * t ? X::abs_(Cxl) : T(2) * a * t;
    // the exponents the polynomials see: |a s^2 + B s| <= (|B| + |a| t) t on [0, t] and |t (W + a t)| (gq lives in the weights)
    const T xmain = ((X::abs_(B0) > X::abs_(W) ? X::abs_(B0) : X::abs_(W)) + X::abs_(a) * t) * t;
    const T xsec = sec * t;
    int level = !(xmain <= T(GGP_FAST_MID) && xsec <= T(GGP_FAST_SMALL8)) ? 0
                : (xmain <= T(GGP_FAST_SMALL8) && xsec <= T(GGP_FAST_TINY4)) ? 3
                : (xmain <= T(GGP_FAST_SMALL) && xsec <= T(GGP_FAST_TINY)) ? 2 : 1;
#if defined(__CUDA_ARCH__)
    // the levels are nested (a lower one is valid wherever a higher one is): the lanes of a warp take the lowest level any of
    // them needs, so that a warp runs ONE variant of the sums.  Rules of 6 nodes and more only: their steps straddle the 0.125
    // threshold (configs[2]: 40 % of the warps ran two variants, 1.04 -> 0.93 ms); a 5-node rule accepts no exponent above 0.12
    // and the reduction costs 4 % where the lanes agree anyway (configs[1]: 0.592 vs 0.569 ms)
    if (N >= 6) level = __reduce_min_sync(__activemask(), level);
#endif
    const T xh = t * (W + a * t);
    const T EH = level == 3 ? X::exp_small8_(xh) : level == 2 ? X::exp_small_(xh) : level == 1 ? X::exp_mid_(xh) : X::exp_(xh);
    T M[12];
    if (level == 3) ggp_fast_moments<T, N, 3>(K, a, B0, Cxl, EH, M);
    else if (level == 2) ggp_fast_moments<T, N, 2>(K, a, B0, Cxl, EH, M);
    else if (level == 1) ggp_fast_moments<T, N, 1>(K, a, B0, Cxl, EH, M);
    else ggp_fast_moments<T, N, 0>(K, a, B0, Cxl, EH, M);
    // exp(c): c0 = bx + Cxx/2 - b t (B-family, mean_cov_model.h:76-115), c5 = 2 (bx + Cxx - b t) (W-family, :124-164)
    const T E1 = X::exp_(bx + T(0.5) * Cxx);
    const T Ec0 = E1 * K.ebt;
    const T aCxx = X::abs_(Cxx);
    const T Ec5 = (E1 * K.ebt) * (E1 * K.ebt) * (aCxx <= T(GGP_FAST_TINY) ? X::exp_tiny_(Cxx) : aCxx <= T(GGP_FAST_MID) ? X::exp_mid_(Cxx) : X::exp_(Cxx));
    const T JB0 = Ec0 * M[0], JB1 = Ec0 * M[1];                        // I_k(B0, c0; 0, t)
    const T JBm0 = Ec0 * M[2], JBm1 = Ec0 * M[3], JBm2 = Ec0 * M[4];   // I_k(B0 - gq, c0; 0, t)
    const T JBs0 = Ec0 * M[5];                                         // I_0(B0 + gq, c0) - I_0(B0 - gq, c0)

    const T dq = bq + Cxq - mq;
    const T G1 = mq * JB0 + dq * JBm0 + Clq * JBm1;   // mean_g - bg e^{-bt}, mean_cov_model.h:76-80
    const T G2 = mq * JB1 + dq * JBm1 + Clq * JBm2;
    const T ebt = K.ebt, egl = K.egl, egq = K.egq, oi = K.oi;

    // means, mean_cov_model.h:73-87
    const T nm0 = bx + ml * t + (bl - ml) * oi;
    const T nm1 = bg * ebt + G1;
    const T nm2 = ml + (bl - ml) * egl;
    const T nm3 = mq + (bq - mq) * egq;

    // x row: cov(x_t, .) with x_t = x_0 + int lambda; alpha, beta, gamma = cov(x_t, x_0 / lambda_0 / q_0)
    const T al = Cxx + Cxl * oi, be = Cxl + Cll * oi, ga = Cxq + Clq * oi;
    const T n_xx = Cxx + T(2) * Cxl * oi + Cll * (oi * oi) + K.kxx;           // :93-95
    const T n_xg = ebt * (Cxg + Cgl * oi) + al * G1 + be * G2 + ga * JBm0;    // :97-115, central form
    const T n_xl = be * egl + K.kxl;                                          // :117-119
    const T n_xq = ga * egq;                                                  // :120-122
    // lambda and q rows
    const T n_gl = egl * (ebt * Cgl + Cxl * G1 + Cll * G2 + Clq * JBm0);      // :166-176, central form
    const T n_gq = egq * (ebt * Cgq + Cxq * G1 + Clq * G2 + Cqq * JBm0 + K.hsq * JBs0);   // :178-192, central form
    const T n_ll = Cll * (egl * egl) + K.kll;                                 // :196-198
    const T n_lq = Clq * egl * egq;                                           // :200-202
    const T n_qq = Cqq * (egq * egq) + K.kqq;                                 // :204-208
    // cov_gg, :124-164: C_gg e^{-2bt} + 2 e^{-bt} cov(g_0, production) + E[production^2] - G1^2
    // E[production^2] = exp(c5) sum_m mono_m Z_m over the monomials 1, Clq, e2, e2^2 + Cqq, Clq e2, Clq^2 (GgpFastNode)
    const T e2 = bq + T(2) * Cxq - mq;
    const T S2 = Ec5 * ((M[6] + Cqq * M[9]) + Clq * (M[7] + e2 * M[10] + Clq * M[11]) + e2 * (M[8] + e2 * M[9]));
    const T n_gg = Cgg * (ebt * ebt) + T(2) * ebt * (Cxg * G1 + Cgl * G2 + Cgq * JBm0) + (S2 - G1 * G1);

    st.m[0] = nm0; st.m[1] = nm1; st.m[2] = nm2; st.m[3] = nm3;
    st.c[0] = n_xx; st.c[1] = n_xg; st.c[2] = n_xl; st.c[3] = n_xq; st.c[4] = n_gg;
    st.c[5] = n_gl; st.c[6] = n_gq; st.c[7] = n_ll; st.c[8] = n_lq; st.c[9] = n_qq;
    return ok;
}

// measurement update (predictions.h:84-89) and the log-evidence term of likelihood.h:26-32 in two parts: returns the quadratic
// form -1/2 r^T S^-1 r and multiplies det S into `pdet`; the caller takes ONE logarithm of the running product per cell
// (sum of log det = log of the product; the product is folded into `lsum` before it can leave the double range).
template <class T>
GGP_HD T ggp_fast_update(GgpFastState<T>& s, T x, T g, T var_x, T var_g, bool noise_scaled, T fp_auto, T& pdet, T& lsum, bool& valid) {
    typedef GgpFx<T> X;
    const T r0 = x - s.m[0], r1 = g - s.m[1];
    const T D11 = noise_scaled ? var_g * (s.m[1] + fp_auto) : var_g;
    const T S00 = s.c[0] + var_x, S01 = s.c[1], S11 = s.c[4] + D11;
    const T det = S00 * S11 - S01 * S01;
    if (!(det > T(0))) valid = false;   // log of a non-positive determinant: NaN in the reference; the strict path reports it
    pdet *= det;
    if (!(pdet < T(1e100) && pdet > T(1e-100))) {
        lsum += X::log_(pdet);
        pdet = T(1);
    }
    const T id = T(1) / det;
    const T Si00 = S11 * id, Si01 = -S01 * id, Si11 = S00 * id;
    const T q0 = Si00 * r0 + Si01 * r1, q1 = Si01 * r0 + Si11 * r1;   // Si r
    const T qf = T(-0.5) * (r0 * q0 + r1 * q1);
    // K = C[0:2, :]: rows (xx xg xl xq), (xg gg gl gq); T_i = K_i^T Si
    const T K0[4] = {s.c[0], s.c[1], s.c[2], s.c[3]};
    const T K1[4] = {s.c[1], s.c[4], s.c[5], s.c[6]};
    T T0[4], T1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        T0[i] = K0[i] * Si00 + K1[i] * Si01;
        T1[i] = K0[i] * Si01 + K1[i] * Si11;
    }
    s.m[0] += K0[0] * q0 + K1[0] * q1;   // m += K^T Si r
    s.m[1] += K0[1] * q0 + K1[1] * q1;
    s.m[2] += K0[2] * q0 + K1[2] * q1;
    s.m[3] += K0[3] * q0 + K1[3] * q1;
    T n[10];
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
    return qf;
}

// mother's last posterior, already propagated over the gap -> daughter's prior (predictions.h:18-61)
template <class T>
GGP_HD void ggp_fast_divide(GgpFastState<T>& s, T var_dx, T var_dg, bool binomial) {
    if (binomial) {
        const T c01 = s.m[1] * T(0.5) * var_dx + s.c[1];
        const T c11 = var_dx * (s.m[1] * s.m[1] + s.c[4]) * T(0.5) + var_dg * s.m[1] * T(0.25) * (T(1) - var_dx) + s.c[4] * T(0.25);
        s.c[0] += var_dx; s.c[1] = c01; s.c[4] = c11;
        s.c[5] *= T(0.5); s.c[6] *= T(0.5);
    } else {
        s.c[0] += var_dx; s.c[1] *= T(0.5); s.c[4] = var_dg + T(0.25) * s.c[4];
        s.c[5] *= T(0.5); s.c[6] *= T(0.5);
    }
    s.m[0] -= GgpFx<T>::ln2();
    s.m[1] *= T(0.5);
}

// ---- one cell of the likelihood (sc_likelihood, likelihood.h:36-103), fresh mode ------------------------------------
// s: in = the mother's end-of-cell posterior (ignored for a root), out = this cell's.  Returns the cell's log-evidence sum;
// clears `valid` if a step left the quadrature's range or a term is NaN (the caller then re-runs the vector strictly).
// KP supplies the (parameters, dt)-only constants of the step that ARRIVES at time point k of the forest:
//   const GgpFastConsts<T, N>& KP::at(int64_t k, int64_t from)
// (host checks: recomputed when dt changes; device: a table over the forest's distinct dt values, ggp_fast.cu).
template <class T, int N, class KP>
GGP_HD T ggp_fast_cell(const GgpDevForest& F, int slot, const T* __restrict__ p, GgpFastState<T>& s, KP& kp, bool& valid) {
    const int64_t off = F.s_off[slot];
    const int n = F.s_n[slot];
    const int parent = F.s_parent[slot];
    const bool scaled = F.model.noise_scaled != 0, binomial = F.model.division_binomial != 0;
    const T fp_auto = T(F.model.fp_auto), lmax = T(GgpFastLmax<N>::v());
    T own = T(0), pdet = T(1), lsum = T(0);
    int t;
    int64_t from;
    if (parent < 0) {   // init_sc_distribution, predictions.h:63-78 (first evaluation: off-diagonals are zero)
        s.m[0] = T(F.init_f[0]); s.m[1] = T(F.init_f[1]); s.m[2] = p[0]; s.m[3] = p[3];
#pragma unroll
        for (int i = 0; i < 10; ++i) s.c[i] = T(0);
        s.c[0] = T(F.init_f[2]); s.c[4] = T(F.init_f[3]);
        s.c[7] = p[2] / (T(2) * p[1]);
        s.c[9] = p[5] / (T(2) * p[4]);
        own += ggp_fast_update(s, T(F.x[off]), T(F.g[off]), p[7], p[8], scaled, fp_auto, pdet, lsum, valid);
        t = 0;
        from = off;
    } else {
        t = -1;
        from = F.s_off[parent] + F.s_n[parent] - 1;
    }
    while (t + 1 < n) {
        const int64_t k = off + t + 1;
        const T xk = T(F.x[k]), gk = T(F.g[k]);   // issued before the step's arithmetic
        const GgpFastConsts<T, N>& K = kp.at(k, from);
        if (!ggp_fast_propagate(s, K, p[0], p[1], p[3], p[4], p[5], p[6], lmax)) valid = false;
        if (t < 0) ggp_fast_divide(s, p[9], p[10], binomial);
        ++t;
        from = k;
        own += ggp_fast_update(s, xk, gk, p[7], p[8], scaled, fp_auto, pdet, lsum, valid);
    }
    // sum over the cell's points of -1/2 log det S - 2 log(2 pi) (the constant as likelihood.h:31 writes it)
    own = own - T(0.5) * (lsum + GgpFx<T>::log_(pdet)) - T(n) * T(3.6757541328186907);
    if (own != own) valid = false;
    return own;
}

// constants recomputed whenever dt changes (host checks, any scalar type)
template <class T, int N, class GL>
struct GgpFastConstsOnDemand {
    const GgpDevForest& F;
    const T* p;
    const GL& gln;
    GgpFastConsts<T, N> K;
    bool have = false;
    GgpFastConstsOnDemand(const GgpDevForest& F_, const T* p_, const GL& g_) : F(F_), p(p_), gln(g_) {}
    const GgpFastConsts<T, N>& at(int64_t k, int64_t from) {
        const T dt = T(F.time[k]) - T(F.time[from]);
        if (!have || !(dt == K.t)) ggp_fast_consts(K, dt, p[0], p[1], p[2], p[3], p[4], p[5], p[6], gln);
        have = true;
        return K;
    }
};
