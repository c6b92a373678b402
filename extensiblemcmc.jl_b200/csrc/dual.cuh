// Forward-mode dual numbers for user-defined laws written over their scalar type (with_grad =
// EXTMCMC_USER_GRAD_FORWARD, see include/extmcmc.h): Dual<K> is a value and the K partial derivatives
// of it with respect to the chain's parameters, the device counterpart of ForwardDiff.Dual.  The user's
// templated `set_parameters` / `logpdf` run unchanged on Law<Dual<P>>; the overloads below are found by
// argument-dependent lookup.
//
// The value part of every operation is the very double operation Law<double> code performs, so under
// -fmad=false a gradient sweep computes the log-likelihood bit for bit as the value sweep does.
// Tangents use the computed value where the derivative allows it (exp: d * v).  Conventions where the
// derivative is not defined: fmax / fmin take the tangents of the operand they return, the first one
// on a tie; fabs at +-0 takes sign +1; pow(a, b) takes 0 as the b-partial at a = 0.
//
// There is deliberately no conversion to double: a function without an overload here (lgamma,
// tgamma, ...) or an assignment of a Dual to a double does not compile, and the compiler log names
// the call, instead of silently dropping the derivatives.
//
// NVRTC compiles this file (no standard headers: the math functions are built in); so do nvcc and a
// host C++ compiler, for tests (the includer provides <cmath> and normcdf).
#pragma once
#ifndef __CUDACC__
#ifndef __host__
#define __host__
#endif
#ifndef __device__
#define __device__
#endif
#ifndef __forceinline__
#define __forceinline__ inline
#endif
#endif

namespace extmcmc {

template <int K>
struct Dual {
    static_assert(K >= 1, "Dual needs at least one tangent");
    double v;       // value
    double t[K];    // d v / d th[k]
    __host__ __device__ __forceinline__ Dual() {}
    // a constant: zero tangents (implicit, so that `real e = 0.0;` and double operands work)
    __host__ __device__ __forceinline__ Dual(double x) : v(x) {
#pragma unroll
        for (int k = 0; k < K; ++k) t[k] = 0.0;
    }
};

#define EXTMCMC_DUAL_FN __host__ __device__ __forceinline__

// r = value, r.t = a * x.t
template <int K>
EXTMCMC_DUAL_FN Dual<K> dual_chain(double value, const Dual<K> &x, double a) {
    Dual<K> r;
    r.v = value;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = a * x.t[k];
    return r;
}

// ---- arithmetic -----------------------------------------------------------------------------------
template <int K> EXTMCMC_DUAL_FN Dual<K> operator+(const Dual<K> &a) { return a; }
template <int K> EXTMCMC_DUAL_FN Dual<K> operator-(const Dual<K> &a) {
    Dual<K> r;
    r.v = -a.v;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = -a.t[k];
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator+(const Dual<K> &a, const Dual<K> &b) {
    Dual<K> r;
    r.v = a.v + b.v;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = a.t[k] + b.t[k];
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator+(const Dual<K> &a, double b) {
    Dual<K> r = a;
    r.v = a.v + b;
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator+(double a, const Dual<K> &b) {
    Dual<K> r = b;
    r.v = a + b.v;
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator-(const Dual<K> &a, const Dual<K> &b) {
    Dual<K> r;
    r.v = a.v - b.v;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = a.t[k] - b.t[k];
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator-(const Dual<K> &a, double b) {
    Dual<K> r = a;
    r.v = a.v - b;
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator-(double a, const Dual<K> &b) {
    Dual<K> r;
    r.v = a - b.v;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = -b.t[k];
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator*(const Dual<K> &a, const Dual<K> &b) {
    Dual<K> r;
    r.v = a.v * b.v;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = a.t[k] * b.v + a.v * b.t[k];
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator*(const Dual<K> &a, double b) { return dual_chain(a.v * b, a, b); }
template <int K> EXTMCMC_DUAL_FN Dual<K> operator*(double a, const Dual<K> &b) { return dual_chain(a * b.v, b, a); }
// q = a / b: d q = (d a - q d b) / b
template <int K> EXTMCMC_DUAL_FN Dual<K> operator/(const Dual<K> &a, const Dual<K> &b) {
    Dual<K> r;
    r.v = a.v / b.v;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = (a.t[k] - r.v * b.t[k]) / b.v;
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator/(const Dual<K> &a, double b) {
    Dual<K> r;
    r.v = a.v / b;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = a.t[k] / b;
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> operator/(double a, const Dual<K> &b) {
    Dual<K> r;
    r.v = a / b.v;
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = -(r.v * b.t[k]) / b.v;
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator+=(Dual<K> &a, const Dual<K> &b) { return a = a + b; }
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator+=(Dual<K> &a, double b) { return a = a + b; }
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator-=(Dual<K> &a, const Dual<K> &b) { return a = a - b; }
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator-=(Dual<K> &a, double b) { return a = a - b; }
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator*=(Dual<K> &a, const Dual<K> &b) { return a = a * b; }
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator*=(Dual<K> &a, double b) { return a = a * b; }
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator/=(Dual<K> &a, const Dual<K> &b) { return a = a / b; }
template <int K> EXTMCMC_DUAL_FN Dual<K> &operator/=(Dual<K> &a, double b) { return a = a / b; }

// ---- comparisons (on the value) -------------------------------------------------------------------
#define EXTMCMC_DUAL_CMP(op)                                                                            \
    template <int K> EXTMCMC_DUAL_FN bool operator op(const Dual<K> &a, const Dual<K> &b) { return a.v op b.v; } \
    template <int K> EXTMCMC_DUAL_FN bool operator op(const Dual<K> &a, double b) { return a.v op b; }           \
    template <int K> EXTMCMC_DUAL_FN bool operator op(double a, const Dual<K> &b) { return a op b.v; }
EXTMCMC_DUAL_CMP(<)
EXTMCMC_DUAL_CMP(<=)
EXTMCMC_DUAL_CMP(>)
EXTMCMC_DUAL_CMP(>=)
EXTMCMC_DUAL_CMP(==)
EXTMCMC_DUAL_CMP(!=)
#undef EXTMCMC_DUAL_CMP

template <int K> EXTMCMC_DUAL_FN bool isinf(const Dual<K> &a) { return ::isinf(a.v); }
template <int K> EXTMCMC_DUAL_FN bool isnan(const Dual<K> &a) { return ::isnan(a.v); }
template <int K> EXTMCMC_DUAL_FN bool isfinite(const Dual<K> &a) { return ::isfinite(a.v); }

// ---- elementary functions -------------------------------------------------------------------------
template <int K> EXTMCMC_DUAL_FN Dual<K> exp(const Dual<K> &x) {
    const double v = ::exp(x.v);
    return dual_chain(v, x, v);
}
template <int K> EXTMCMC_DUAL_FN Dual<K> expm1(const Dual<K> &x) {
    const double v = ::expm1(x.v);
    return dual_chain(v, x, v + 1.0);
}
template <int K> EXTMCMC_DUAL_FN Dual<K> log(const Dual<K> &x) { return dual_chain(::log(x.v), x, 1.0 / x.v); }
template <int K> EXTMCMC_DUAL_FN Dual<K> log1p(const Dual<K> &x) { return dual_chain(::log1p(x.v), x, 1.0 / (1.0 + x.v)); }
template <int K> EXTMCMC_DUAL_FN Dual<K> sqrt(const Dual<K> &x) {
    const double v = ::sqrt(x.v);
    return dual_chain(v, x, 0.5 / v);
}
template <int K> EXTMCMC_DUAL_FN Dual<K> pow(const Dual<K> &x, double p) {
    return dual_chain(::pow(x.v, p), x, p * ::pow(x.v, p - 1.0));
}
template <int K> EXTMCMC_DUAL_FN Dual<K> pow(double a, const Dual<K> &p) {
    const double v = ::pow(a, p.v);
    return dual_chain(v, p, a == 0.0 ? 0.0 : v * ::log(a));
}
// d a^b = b a^(b-1) d a + a^b log(a) d b
template <int K> EXTMCMC_DUAL_FN Dual<K> pow(const Dual<K> &a, const Dual<K> &b) {
    Dual<K> r;
    r.v = ::pow(a.v, b.v);
    const double da = b.v * ::pow(a.v, b.v - 1.0), db = a.v == 0.0 ? 0.0 : r.v * ::log(a.v);
#pragma unroll
    for (int k = 0; k < K; ++k) r.t[k] = da * a.t[k] + db * b.t[k];
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> fabs(const Dual<K> &x) { return dual_chain(::fabs(x.v), x, x.v < 0.0 ? -1.0 : 1.0); }
template <int K> EXTMCMC_DUAL_FN Dual<K> sin(const Dual<K> &x) { return dual_chain(::sin(x.v), x, ::cos(x.v)); }
template <int K> EXTMCMC_DUAL_FN Dual<K> cos(const Dual<K> &x) { return dual_chain(::cos(x.v), x, -::sin(x.v)); }
// 1 - tanh^2 loses digits for large |x|: 1 / cosh^2 does not
template <int K> EXTMCMC_DUAL_FN Dual<K> tanh(const Dual<K> &x) {
    const double c = ::cosh(x.v);
    return dual_chain(::tanh(x.v), x, 1.0 / (c * c));
}
// 2 / sqrt(pi) and 1 / sqrt(2 pi)
template <int K> EXTMCMC_DUAL_FN Dual<K> erf(const Dual<K> &x) {
    return dual_chain(::erf(x.v), x, 1.1283791670955126 * ::exp(-(x.v * x.v)));
}
template <int K> EXTMCMC_DUAL_FN Dual<K> erfc(const Dual<K> &x) {
    return dual_chain(::erfc(x.v), x, -1.1283791670955126 * ::exp(-(x.v * x.v)));
}
template <int K> EXTMCMC_DUAL_FN Dual<K> normcdf(const Dual<K> &x) {
    return dual_chain(::normcdf(x.v), x, 0.3989422804014327 * ::exp(-0.5 * (x.v * x.v)));
}

// fmax / fmin: the value of the double call, the tangents of the operand it returns (the first one on
// a tie; the other one when an operand is NaN, as the double call returns it)
template <int K> EXTMCMC_DUAL_FN Dual<K> fmax(const Dual<K> &a, const Dual<K> &b) {
    Dual<K> r = (a.v >= b.v || b.v != b.v) ? a : b;
    r.v = ::fmax(a.v, b.v);
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> fmax(const Dual<K> &a, double b) {
    Dual<K> r = (a.v >= b || b != b) ? a : Dual<K>(b);
    r.v = ::fmax(a.v, b);
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> fmax(double a, const Dual<K> &b) {
    Dual<K> r = (a >= b.v || b.v != b.v) ? Dual<K>(a) : b;
    r.v = ::fmax(a, b.v);
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> fmin(const Dual<K> &a, const Dual<K> &b) {
    Dual<K> r = (a.v <= b.v || b.v != b.v) ? a : b;
    r.v = ::fmin(a.v, b.v);
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> fmin(const Dual<K> &a, double b) {
    Dual<K> r = (a.v <= b || b != b) ? a : Dual<K>(b);
    r.v = ::fmin(a.v, b);
    return r;
}
template <int K> EXTMCMC_DUAL_FN Dual<K> fmin(double a, const Dual<K> &b) {
    Dual<K> r = (a <= b.v || b.v != b.v) ? Dual<K>(a) : b;
    r.v = ::fmin(a, b.v);
    return r;
}

// fma(a, b, c) = a b + c, rounded once; every combination with at least one Dual operand
template <class T> struct dual_k { static constexpr int value = 0; };
template <int K> struct dual_k<Dual<K>> { static constexpr int value = K; };
template <bool B, int K> struct dual_if {};
template <int K> struct dual_if<true, K> { typedef Dual<K> type; };
template <class T> EXTMCMC_DUAL_FN double dual_val(const T &x) { return x; }
template <int K> EXTMCMC_DUAL_FN double dual_val(const Dual<K> &x) { return x.v; }

template <class A, class B, class C,
          int K = dual_k<A>::value ? dual_k<A>::value : dual_k<B>::value ? dual_k<B>::value : dual_k<C>::value>
EXTMCMC_DUAL_FN typename dual_if<(K > 0) && (!dual_k<A>::value || dual_k<A>::value == K) &&
                                      (!dual_k<B>::value || dual_k<B>::value == K) &&
                                      (!dual_k<C>::value || dual_k<C>::value == K), K>::type
fma(const A &a, const B &b, const C &c) {
    Dual<K> r;
    r.v = ::fma(dual_val(a), dual_val(b), dual_val(c));
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double s = 0.0;
        if constexpr (dual_k<A>::value != 0) s = s + a.t[k] * dual_val(b);
        if constexpr (dual_k<B>::value != 0) s = s + dual_val(a) * b.t[k];
        if constexpr (dual_k<C>::value != 0) s = s + c.t[k];
        r.t[k] = s;
    }
    return r;
}

#undef EXTMCMC_DUAL_FN

}  // namespace extmcmc
