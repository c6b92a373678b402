"""The sample laws of tests/user_laws.py restated for forward-mode gradients (with_grad =
EXTMCMC_USER_GRAD_FORWARD, DeviceLaw(..., gradient="forward")): written once, generic over their
scalar `real`, without logpdf_grad.  The numpy references of tests/user_laws.py apply unchanged.  Also
two sources that must not compile in forward mode."""
from tests import user_laws as ul

GSN1D = r"""
template <class real> struct Law { real mu, c0, h; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    const real var = th[1];
    if (!(var > 0.0) || isinf(var)) return false;
    L.mu = th[0];
    L.c0 = -(1.8378770664093453 + 2.0 * log(sqrt(var))) / 2.0;
    L.h = 0.5 / var;
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    const real d = x[0] - L.mu;
    return L.c0 - d * d * L.h;
}
"""

LOGISTIC = r"""
template <class real> struct Law { real b[EXTMCMC_P]; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    for (int k = 0; k < EXTMCMC_P; ++k) L.b[k] = th[k];
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    real e = 0.0;
    for (int k = 0; k < EXTMCMC_P; ++k) e += x[k] * L.b[k];
    return x[EXTMCMC_P] * e - (fmax(e, 0.0) + log1p(exp(-fabs(e))));
}
"""

POISSON_REG = r"""
template <class real> struct Law { real b[EXTMCMC_P]; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    for (int k = 0; k < EXTMCMC_P; ++k) L.b[k] = th[k];
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    real e = L.b[0];
    for (int k = 1; k < EXTMCMC_P; ++k) e += x[k - 1] * L.b[k];
    return x[EXTMCMC_D - 1] * e - exp(e);
}
"""

POISSON_RATE = r"""
template <class real> struct Law { real lam, loglam; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    if (!(th[0] > 0.0)) return false;
    L.lam = th[0];
    L.loglam = log(th[0]);
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    return x[0] * L.loglam - L.lam;
}
"""

# a function Dual has no overload for: the complete Poisson log-likelihood with -lgamma(y + 1) applied
# to the rate instead of the count (a bug a hand-written gradient would hide)
BAD_LGAMMA = POISSON_RATE.replace("return x[0] * L.loglam - L.lam;",
                                  "return x[0] * L.loglam - L.lam - lgamma(L.lam + 1.0);")
# a real narrowed to double: the derivative would be lost silently
BAD_NARROW = POISSON_RATE.replace("return x[0] * L.loglam - L.lam;",
                                  "const double lam = L.lam;\n    return x[0] * L.loglam - lam;")


def poisson_rate_terms(theta, X, dtype=None):
    import numpy as np
    dtype = dtype or np.float64
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    lam = theta[0][None, :]
    t = X[:, :1] * np.log(lam) - lam
    g = (X[:, :1] / lam - 1.0)[None]
    return t, g


# name -> (forward source, hand-gradient source or None, P(D), terms)
LAWS = {
    "gsn1d": (GSN1D, ul.GSN1D, ul.LAWS["gsn1d"][1], ul.LAWS["gsn1d"][2]),
    "logistic": (LOGISTIC, ul.LOGISTIC, ul.LAWS["logistic"][1], ul.LAWS["logistic"][2]),
    "poisson_reg": (POISSON_REG, ul.POISSON_REG, ul.LAWS["poisson_reg"][1], ul.LAWS["poisson_reg"][2]),
    "poisson_rate": (POISSON_RATE, None, lambda D: 1, poisson_rate_terms),
}
