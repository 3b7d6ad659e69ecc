// ggp_dual.cuh — forward-mode dual numbers for the FAST likelihood step (ggp_fast.cuh), host and device.
//
// GgpDual<D> carries a value and D tangents (derivatives along D parameter directions).  ggp_fast.cuh is templated on its
// scalar type, so ggp_fast_cell<GgpDual<D>, N> evaluates the fast log-likelihood and its derivatives along the seeded
// directions in one pass, without a change to the step's code:
//   * arithmetic propagates the tangents by the product / quotient rules;
//   * comparisons and finite_ read the value only: they choose branches (validity checks, Taylor levels, the rescaling of the
//     running determinant product) and are not part of the result;
//   * each short Taylor exponential of GgpFx<double> is its own derivative (exp' = exp): the tangent is the polynomial's value
//     times the argument's tangent, so the derivative's error is the polynomial's truncation error (at most 3e-17 relative).
// The strict path has no gradient: its purpose is the reference's rounding, whose derivative means nothing.
#pragma once
#include "ggp_fast.cuh"

template <int D>
struct GgpDual {
    double v;      // value
    double d[D];   // tangents
    GgpDual() = default;
    GGP_HDM GgpDual(double x) : v(x) {   // a constant: zero tangents
#pragma unroll
        for (int i = 0; i < D; ++i) d[i] = 0.0;
    }
};

template <int D>
GGP_HDM GgpDual<D> operator-(const GgpDual<D>& a) {
    GgpDual<D> r;
    r.v = -a.v;
#pragma unroll
    for (int i = 0; i < D; ++i) r.d[i] = -a.d[i];
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator+(const GgpDual<D>& a, const GgpDual<D>& b) {
    GgpDual<D> r;
    r.v = a.v + b.v;
#pragma unroll
    for (int i = 0; i < D; ++i) r.d[i] = a.d[i] + b.d[i];
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator-(const GgpDual<D>& a, const GgpDual<D>& b) {
    GgpDual<D> r;
    r.v = a.v - b.v;
#pragma unroll
    for (int i = 0; i < D; ++i) r.d[i] = a.d[i] - b.d[i];
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator*(const GgpDual<D>& a, const GgpDual<D>& b) {
    GgpDual<D> r;
    r.v = a.v * b.v;
#pragma unroll
    for (int i = 0; i < D; ++i) r.d[i] = a.v * b.d[i] + a.d[i] * b.v;
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator/(const GgpDual<D>& a, const GgpDual<D>& b) {
    GgpDual<D> r;
    r.v = a.v / b.v;
    const double ib = 1.0 / b.v;
#pragma unroll
    for (int i = 0; i < D; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * ib;
    return r;
}
// with a constant on either side
template <int D>
GGP_HDM GgpDual<D> operator+(const GgpDual<D>& a, double b) {
    GgpDual<D> r = a;
    r.v = a.v + b;
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator+(double a, const GgpDual<D>& b) { return b + a; }
template <int D>
GGP_HDM GgpDual<D> operator-(const GgpDual<D>& a, double b) {
    GgpDual<D> r = a;
    r.v = a.v - b;
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator-(double a, const GgpDual<D>& b) {
    GgpDual<D> r = -b;
    r.v = a - b.v;
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator*(const GgpDual<D>& a, double b) {
    GgpDual<D> r;
    r.v = a.v * b;
#pragma unroll
    for (int i = 0; i < D; ++i) r.d[i] = a.d[i] * b;
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator*(double a, const GgpDual<D>& b) { return b * a; }
template <int D>
GGP_HDM GgpDual<D> operator/(const GgpDual<D>& a, double b) {
    GgpDual<D> r;
    r.v = a.v / b;
    const double ib = 1.0 / b;
#pragma unroll
    for (int i = 0; i < D; ++i) r.d[i] = a.d[i] * ib;
    return r;
}
template <int D>
GGP_HDM GgpDual<D> operator/(double a, const GgpDual<D>& b) { return GgpDual<D>(a) / b; }

template <int D>
GGP_HDM GgpDual<D>& operator+=(GgpDual<D>& a, const GgpDual<D>& b) { return a = a + b; }
template <int D>
GGP_HDM GgpDual<D>& operator-=(GgpDual<D>& a, const GgpDual<D>& b) { return a = a - b; }
template <int D>
GGP_HDM GgpDual<D>& operator*=(GgpDual<D>& a, const GgpDual<D>& b) { return a = a * b; }
template <int D>
GGP_HDM GgpDual<D>& operator/=(GgpDual<D>& a, const GgpDual<D>& b) { return a = a / b; }

// comparisons: the value part only
#define GGP_DUAL_CMP(OP)                                                                                  \
    template <int D> GGP_HDM bool operator OP(const GgpDual<D>& a, const GgpDual<D>& b) { return a.v OP b.v; } \
    template <int D> GGP_HDM bool operator OP(const GgpDual<D>& a, double b) { return a.v OP b; }             \
    template <int D> GGP_HDM bool operator OP(double a, const GgpDual<D>& b) { return a OP b.v; }
GGP_DUAL_CMP(<)
GGP_DUAL_CMP(<=)
GGP_DUAL_CMP(>)
GGP_DUAL_CMP(>=)
GGP_DUAL_CMP(==)
GGP_DUAL_CMP(!=)
#undef GGP_DUAL_CMP

template <int D>
struct GgpFx<GgpDual<D>> {
    typedef GgpDual<D> T;
    typedef GgpFx<double> X;
    // f(a) with f'(a) = df: value fa, tangents df * a.d
    static GGP_HDM T chain_(const T& a, double fa, double df) {
        T r;
        r.v = fa;
#pragma unroll
        for (int i = 0; i < D; ++i) r.d[i] = df * a.d[i];
        return r;
    }
    static GGP_HDM T exp_(const T& x) { const double e = X::exp_(x.v); return chain_(x, e, e); }
    static GGP_HDM T log_(const T& x) { return chain_(x, X::log_(x.v), 1.0 / x.v); }
    static GGP_HDM T expm1_(const T& x) { const double e = X::expm1_(x.v); return chain_(x, e, e + 1.0); }
    static GGP_HDM T abs_(const T& x) { return x.v < 0.0 ? -x : x; }
    static GGP_HDM bool finite_(const T& x) { return X::finite_(x.v); }
    static GGP_HDM T ln2() { return T(X::ln2()); }
    // the Taylor exponentials: the polynomial's value is its own derivative
    template <int DEG>
    static GGP_HDM T exp_taylor_(const T& x) { const double e = X::template exp_taylor_<DEG>(x.v); return chain_(x, e, e); }
    static GGP_HDM T exp_mid_(const T& x) { return exp_taylor_<15>(x); }
    static GGP_HDM T exp_small_(const T& x) { return exp_taylor_<10>(x); }
    static GGP_HDM T exp_small8_(const T& x) { return exp_taylor_<8>(x); }
    static GGP_HDM T exp_tiny_(const T& x) { return exp_taylor_<6>(x); }
    static GGP_HDM T exp_tiny4_(const T& x) { return exp_taylor_<4>(x); }
};

// ---- GgpTaylor2: the truncated Taylor series of order 2 along one direction u ----------------------------------------------
// (v, d, dd) = (f, f' u, u^T f'' u) of a function f of the parameters, carried through the fast step like GgpDual: one
// evaluation seeded with u returns the value, the directional derivative g.u and the quadratic form u^T H u of the
// log-likelihood.  The mixed second derivatives come from several directions by polarization (DESIGN.md 5.7).  Comparisons
// and finite_ read the value only, as for GgpDual.
struct GgpTaylor2 {
    double v, d, dd;
    GgpTaylor2() = default;
    GGP_HDM GgpTaylor2(double x) : v(x), d(0.0), dd(0.0) {}   // a constant
    GGP_HDM GgpTaylor2(double x, double dx, double ddx) : v(x), d(dx), dd(ddx) {}
};

GGP_HDM GgpTaylor2 operator-(const GgpTaylor2& a) { return GgpTaylor2(-a.v, -a.d, -a.dd); }
GGP_HDM GgpTaylor2 operator+(const GgpTaylor2& a, const GgpTaylor2& b) { return GgpTaylor2(a.v + b.v, a.d + b.d, a.dd + b.dd); }
GGP_HDM GgpTaylor2 operator-(const GgpTaylor2& a, const GgpTaylor2& b) { return GgpTaylor2(a.v - b.v, a.d - b.d, a.dd - b.dd); }
GGP_HDM GgpTaylor2 operator*(const GgpTaylor2& a, const GgpTaylor2& b) {
    return GgpTaylor2(a.v * b.v, a.v * b.d + a.d * b.v, a.v * b.dd + 2.0 * (a.d * b.d) + a.dd * b.v);
}
GGP_HDM GgpTaylor2 operator/(const GgpTaylor2& a, const GgpTaylor2& b) {
    const double ib = 1.0 / b.v;
    const double r = a.v / b.v;
    const double rd = (a.d - r * b.d) * ib;
    return GgpTaylor2(r, rd, (a.dd - r * b.dd - 2.0 * (rd * b.d)) * ib);
}
// with a constant on either side
GGP_HDM GgpTaylor2 operator+(const GgpTaylor2& a, double b) { return GgpTaylor2(a.v + b, a.d, a.dd); }
GGP_HDM GgpTaylor2 operator+(double a, const GgpTaylor2& b) { return b + a; }
GGP_HDM GgpTaylor2 operator-(const GgpTaylor2& a, double b) { return GgpTaylor2(a.v - b, a.d, a.dd); }
GGP_HDM GgpTaylor2 operator-(double a, const GgpTaylor2& b) { return GgpTaylor2(a - b.v, -b.d, -b.dd); }
GGP_HDM GgpTaylor2 operator*(const GgpTaylor2& a, double b) { return GgpTaylor2(a.v * b, a.d * b, a.dd * b); }
GGP_HDM GgpTaylor2 operator*(double a, const GgpTaylor2& b) { return b * a; }
GGP_HDM GgpTaylor2 operator/(const GgpTaylor2& a, double b) {
    const double ib = 1.0 / b;
    return GgpTaylor2(a.v / b, a.d * ib, a.dd * ib);
}
GGP_HDM GgpTaylor2 operator/(double a, const GgpTaylor2& b) { return GgpTaylor2(a) / b; }

GGP_HDM GgpTaylor2& operator+=(GgpTaylor2& a, const GgpTaylor2& b) { return a = a + b; }
GGP_HDM GgpTaylor2& operator-=(GgpTaylor2& a, const GgpTaylor2& b) { return a = a - b; }
GGP_HDM GgpTaylor2& operator*=(GgpTaylor2& a, const GgpTaylor2& b) { return a = a * b; }
GGP_HDM GgpTaylor2& operator/=(GgpTaylor2& a, const GgpTaylor2& b) { return a = a / b; }

// comparisons: the value part only
#define GGP_TAYLOR2_CMP(OP)                                                                     \
    GGP_HDM bool operator OP(const GgpTaylor2& a, const GgpTaylor2& b) { return a.v OP b.v; } \
    GGP_HDM bool operator OP(const GgpTaylor2& a, double b) { return a.v OP b; }             \
    GGP_HDM bool operator OP(double a, const GgpTaylor2& b) { return a OP b.v; }
GGP_TAYLOR2_CMP(<)
GGP_TAYLOR2_CMP(<=)
GGP_TAYLOR2_CMP(>)
GGP_TAYLOR2_CMP(>=)
GGP_TAYLOR2_CMP(==)
GGP_TAYLOR2_CMP(!=)
#undef GGP_TAYLOR2_CMP

template <>
struct GgpFx<GgpTaylor2> {
    typedef GgpTaylor2 T;
    typedef GgpFx<double> X;
    // f(a) with f'(a) = df, f''(a) = ddf: (fa, df a.d, df a.dd + ddf a.d^2)
    static GGP_HDM T chain_(const T& a, double fa, double df, double ddf) { return T(fa, df * a.d, df * a.dd + ddf * (a.d * a.d)); }
    static GGP_HDM T exp_(const T& x) { const double e = X::exp_(x.v); return chain_(x, e, e, e); }
    static GGP_HDM T log_(const T& x) { const double r = 1.0 / x.v; return chain_(x, X::log_(x.v), r, -(r * r)); }
    static GGP_HDM T expm1_(const T& x) { const double e = X::expm1_(x.v); return chain_(x, e, e + 1.0, e + 1.0); }
    static GGP_HDM T abs_(const T& x) { return x.v < 0.0 ? -x : x; }
    static GGP_HDM bool finite_(const T& x) { return X::finite_(x.v); }
    static GGP_HDM T ln2() { return T(X::ln2()); }
    // the Taylor exponentials: the polynomial's value is its own first and second derivative
    template <int DEG>
    static GGP_HDM T exp_taylor_(const T& x) { const double e = X::template exp_taylor_<DEG>(x.v); return chain_(x, e, e, e); }
    static GGP_HDM T exp_mid_(const T& x) { return exp_taylor_<15>(x); }
    static GGP_HDM T exp_small_(const T& x) { return exp_taylor_<10>(x); }
    static GGP_HDM T exp_small8_(const T& x) { return exp_taylor_<8>(x); }
    static GGP_HDM T exp_tiny_(const T& x) { return exp_taylor_<6>(x); }
    static GGP_HDM T exp_tiny4_(const T& x) { return exp_taylor_<4>(x); }
};
