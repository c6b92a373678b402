"""Sources of the device laws the user-law tests and tools/user_law_bench.py use (CUDA C++, the
contract of include/extmcmc.h), with numpy references of their per-row terms and gradients (fp64 by
default; dtype=np.longdouble gives the extended-precision reference)."""
import numpy as np

LOG2PI = 1.8378770664093453

# GsnTargetLaw, d = 1 (src/example/gsn_target.jl), theta = [mu, sigma^2]: the expressions of the
# built-in GSN_IID_1D law's constants, one row at a time
GSN1D = r"""
struct Law { double mu, c0, h; };
__device__ bool set_parameters(Law &L, const double *th) {
    const double var = th[1];
    if (!(var > 0.0) || isinf(var)) return false;    // Normal(mu, sqrt(var)) throws there
    L.mu = th[0];
    L.c0 = -(1.8378770664093453 + 2.0 * log(sqrt(var))) / 2.0;
    L.h = 0.5 / var;
    return true;
}
__device__ double logpdf(const Law &L, const double *x) {
    const double d = x[0] - L.mu;
    return L.c0 - d * d * L.h;
}
__device__ double logpdf_grad(const Law &L, const double *x, double *g) {
    const double d = x[0] - L.mu;
    g[0] += 2.0 * L.h * d;                           // d / dmu  =  (x - mu) / var
    g[1] += 2.0 * L.h * L.h * (d * d) - L.h;         // d / dvar = (x - mu)^2 / (2 var^2) - 1 / (2 var)
    return L.c0 - d * d * L.h;
}
"""

# Bayesian logistic regression without intercept: theta = beta[P], row = [x_1..x_P, y], D = P + 1
LOGISTIC = r"""
struct Law { double b[EXTMCMC_P]; };
__device__ bool set_parameters(Law &L, const double *th) {
    for (int k = 0; k < EXTMCMC_P; ++k) L.b[k] = th[k];
    return true;
}
__device__ double eta(const Law &L, const double *x) {
    double e = 0.0;
    for (int k = 0; k < EXTMCMC_P; ++k) e += x[k] * L.b[k];
    return e;
}
__device__ double logpdf(const Law &L, const double *x) {
    const double e = eta(L, x);
    return x[EXTMCMC_P] * e - (fmax(e, 0.0) + log1p(exp(-fabs(e))));    // y e - log(1 + e^e)
}
__device__ double logpdf_grad(const Law &L, const double *x, double *g) {
    const double e = eta(L, x), r = x[EXTMCMC_P] - 1.0 / (1.0 + exp(-e));
    for (int k = 0; k < EXTMCMC_P; ++k) g[k] += r * x[k];
    return x[EXTMCMC_P] * e - (fmax(e, 0.0) + log1p(exp(-fabs(e))));
}
"""

# Poisson regression with log link and intercept: theta = beta[P], row = [x_1..x_{P-1}, y], D = P;
# the log-likelihood up to its theta-free term -lgamma(y + 1)
POISSON_REG = r"""
struct Law { double b[EXTMCMC_P]; };
__device__ bool set_parameters(Law &L, const double *th) {
    for (int k = 0; k < EXTMCMC_P; ++k) L.b[k] = th[k];
    return true;
}
__device__ double lin(const Law &L, const double *x) {
    double e = L.b[0];
    for (int k = 1; k < EXTMCMC_P; ++k) e += x[k - 1] * L.b[k];
    return e;
}
__device__ double logpdf(const Law &L, const double *x) {
    const double y = x[EXTMCMC_D - 1], e = lin(L, x);
    return y * e - exp(e);
}
__device__ double logpdf_grad(const Law &L, const double *x, double *g) {
    const double y = x[EXTMCMC_D - 1], e = lin(L, x), r = y - exp(e);
    g[0] += r;
    for (int k = 1; k < EXTMCMC_P; ++k) g[k] += r * x[k - 1];
    return y * e - exp(e);
}
"""

# Poisson counts with their rate as the parameter: theta = [lambda], row = [y] (up to -lgamma(y + 1))
POISSON_RATE = r"""
struct Law { double lam, loglam; };
__device__ bool set_parameters(Law &L, const double *th) {
    if (!(th[0] > 0.0)) return false;
    L.lam = th[0];
    L.loglam = log(th[0]);
    return true;
}
__device__ double logpdf(const Law &L, const double *x) {
    return x[0] * L.loglam - L.lam;
}
"""


def gsn1d_terms(theta, X, dtype=np.float64):
    """[N, C] per-row log-densities and [P, N, C] gradients; theta [2, C], X [N, 1]."""
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    mu, var = theta[0][None, :], theta[1][None, :]
    d = X[:, :1] - mu
    t = -(LOG2PI + np.log(var)) / 2.0 - d * d / (2.0 * var)
    g = np.stack([d / var, d * d / (2.0 * var * var) - 1.0 / (2.0 * var)])
    return t, g


def logistic_terms(theta, X, dtype=np.float64):
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    P = theta.shape[0]
    e = X[:, :P] @ theta
    y = X[:, P:P + 1]
    t = y * e - np.logaddexp(0.0, e)
    r = y - 1.0 / (1.0 + np.exp(-e))
    g = r[None, :, :] * X[:, :P].T[:, :, None]
    return t, g


def poisson_reg_terms(theta, X, dtype=np.float64):
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    P = theta.shape[0]
    e = theta[0][None, :] + X[:, :P - 1] @ theta[1:]
    y = X[:, P - 1:P]
    t = y * e - np.exp(e)
    r = y - np.exp(e)
    g = np.concatenate([r[None], r[None, :, :] * X[:, :P - 1].T[:, :, None]], axis=0)
    return t, g


# name -> (source, P(D), terms); the regression laws take their dimensions from D
LAWS = {
    "gsn1d": (GSN1D, lambda D: 2, gsn1d_terms),
    "logistic": (LOGISTIC, lambda D: D - 1, logistic_terms),
    "poisson_reg": (POISSON_REG, lambda D: D, poisson_reg_terms),
}
