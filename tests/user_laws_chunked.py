"""Forward-mode sample laws for chunked gradients (extmcmc_set_user_law_chunked, DeviceLaw(...,
gradient="forward", chunk=...)) at large P, beside the templated Poisson regression and logistic sources
of tests/user_laws_forward.py: a law whose every field carries a live tangent (positive coefficients
w_k = exp(th_k)), a Gaussian linear regression with known sigma, and a regression with its scale as a
parameter, whose set_parameters fails at sigma <= 0.  numpy references of the per-row terms and
gradients as in tests/user_laws.py (dtype=np.longdouble: extended precision), and data / state
generators."""
import math

import numpy as np

from tests import user_laws as ul
from tests import user_laws_forward as uf

LOG2PI = ul.LOG2PI
SIGMA = 0.5          # the known noise scale of GAUSS_REG

# Linear regression with positive coefficients w_k = exp(th_k) and unit noise: mean w_0 +
# sum_k w_k x_k, row = [x_1..x_{P-1}, y], D = P (up to its theta-free constant).  set_parameters leaves
# no field a copy of theta: every w_k holds K live tangents in a chunk of width K.
POS_REG = r"""
template <class real> struct Law { real w[EXTMCMC_P]; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    for (int k = 0; k < EXTMCMC_P; ++k) L.w[k] = exp(th[k]);
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    real m = L.w[0];
    for (int k = 1; k < EXTMCMC_P; ++k) m += x[k - 1] * L.w[k];
    const real d = x[EXTMCMC_D - 1] - m;
    return -0.5 * (d * d);
}
"""

# Gaussian linear regression with intercept and known sigma = 0.5: theta = beta[P],
# row = [x_1..x_{P-1}, y], D = P
GAUSS_REG = r"""
template <class real> struct Law { real b[EXTMCMC_P]; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    for (int k = 0; k < EXTMCMC_P; ++k) L.b[k] = th[k];
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    real m = L.b[0];
    for (int k = 1; k < EXTMCMC_P; ++k) m += x[k - 1] * L.b[k];
    const real r = (x[EXTMCMC_D - 1] - m) / 0.5;
    return -0.5 * (r * r) - (0.91893853320467267 + log(0.5));
}
"""

# Gaussian linear regression with intercept and unknown scale: theta = [beta_0..beta_{P-2}, sigma],
# row = [x_1..x_{P-2}, y], D = P - 1; set_parameters fails at sigma <= 0
GAUSS_REG_SCALE = r"""
template <class real> struct Law { real b[EXTMCMC_P - 1]; real h, c0; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    const real s = th[EXTMCMC_P - 1];
    if (!(s > 0.0) || isinf(s)) return false;
    for (int k = 0; k < EXTMCMC_P - 1; ++k) L.b[k] = th[k];
    L.h = 0.5 / (s * s);
    L.c0 = -(0.91893853320467267 + log(s));
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    real m = L.b[0];
    for (int k = 1; k < EXTMCMC_P - 1; ++k) m += x[k - 1] * L.b[k];
    const real d = x[EXTMCMC_D - 1] - m;
    return L.c0 - d * d * L.h;
}
"""


def pos_reg_terms(theta, X, dtype=np.float64):
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    P = theta.shape[0]
    w = np.exp(theta)
    m = w[0][None, :] + X[:, :P - 1] @ w[1:]
    r = X[:, P - 1:P] - m
    t = -0.5 * r * r
    g = np.concatenate([r[None], r[None, :, :] * X[:, :P - 1].T[:, :, None]], axis=0) * w[:, None, :]
    return t, g


def gauss_reg_terms(theta, X, dtype=np.float64):
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    P = theta.shape[0]
    s = dtype(SIGMA)
    m = theta[0][None, :] + X[:, :P - 1] @ theta[1:]
    d = X[:, P - 1:P] - m
    t = -0.5 * (d / s) ** 2 - (dtype(LOG2PI) / 2 + np.log(s))
    r = d / (s * s)
    g = np.concatenate([r[None], r[None, :, :] * X[:, :P - 1].T[:, :, None]], axis=0)
    return t, g


def gauss_reg_scale_terms(theta, X, dtype=np.float64):
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    P = theta.shape[0]
    b, s = theta[:P - 1], theta[P - 1][None, :]
    m = b[0][None, :] + X[:, :P - 2] @ b[1:]
    d = X[:, P - 2:P - 1] - m
    t = -(dtype(LOG2PI) / 2 + np.log(s)) - d * d / (2 * s * s)
    r = d / (s * s)
    gs = d * d / (s * s * s) - 1.0 / s
    g = np.concatenate([r[None], r[None, :, :] * X[:, :P - 2].T[:, :, None], gs[None]], axis=0)
    return t, g


# name -> (forward source, D(P), terms); every law takes P up to 64 except logistic (D = P + 1 <= 64)
LAWS = {
    "poisson_reg": (uf.POISSON_REG, lambda P: P, ul.poisson_reg_terms),
    "logistic": (uf.LOGISTIC, lambda P: P + 1, ul.logistic_terms),
    "pos_reg": (POS_REG, lambda P: P, pos_reg_terms),
    "gauss_reg": (GAUSS_REG, lambda P: P, gauss_reg_terms),
    "gauss_reg_scale": (GAUSS_REG_SCALE, lambda P: P - 1, gauss_reg_scale_terms),
}


def max_params(name):
    return 63 if name == "logistic" else 64


def data(name, N, P, seed=0):
    """Rows [N, D] drawn from the law at a random parameter."""
    rng = np.random.default_rng(seed)
    D = LAWS[name][1](P)
    X = np.empty((N, D))
    if name == "logistic":
        X[:, :P] = rng.standard_normal((N, P)) / math.sqrt(P)
        beta = 0.5 * rng.standard_normal(P)
        X[:, P] = rng.random(N) < 1.0 / (1.0 + np.exp(-X[:, :P] @ beta))
        return X
    nx = D - 1
    X[:, :nx] = rng.standard_normal((N, nx)) / math.sqrt(max(nx, 1))
    if name == "poisson_reg":
        beta = 0.5 * rng.standard_normal(P)
        X[:, nx] = rng.poisson(np.exp(beta[0] + X[:, :nx] @ beta[1:]))
    elif name == "pos_reg":
        w = np.exp(0.3 * rng.standard_normal(P))
        X[:, nx] = w[0] + X[:, :nx] @ w[1:] + rng.standard_normal(N)
    elif name == "gauss_reg":
        beta = rng.standard_normal(P)
        X[:, nx] = beta[0] + X[:, :nx] @ beta[1:] + SIGMA * rng.standard_normal(N)
    else:
        beta = rng.standard_normal(P - 1)
        X[:, nx] = beta[0] + X[:, :nx] @ beta[1:] + 0.7 * rng.standard_normal(N)
    return X


def theta(name, P, Cn, seed=1):
    """A state [P, C] in the law's domain."""
    rng = np.random.default_rng(seed)
    th = 0.3 * rng.standard_normal((P, Cn))
    if name == "gauss_reg_scale":
        th[P - 1] = 0.7 * np.exp(0.1 * rng.standard_normal(Cn))
    return th
