"""Device laws with a term of theta only (flags = EXTMCMC_USER_THETA_TERM, DeviceLaw(...,
theta_term=True)): the hierarchical normal model of BASELINE cfg 4 restated as a user law in plain,
hand-gradient and forward forms, and a Poisson regression with a ridge penalty whose precision appears
in the term only.  numpy references of the per-row terms, the theta term and their gradients
(dtype=np.longdouble: extended precision), data and state generators, and sources that must not compile
with the flag."""
import math

import numpy as np

from tests import user_laws as ul
from tests import user_laws_forward as uf

LOG2PI = ul.LOG2PI
G = 8                # groups of the hierarchical samples: theta = [theta_1..theta_8, mu, tau], P = 10

# Hierarchical normal (the built-in HIER_NORMAL law): theta = [theta_1..theta_G, mu, tau], row = [y, g]
# with g the 0-based group; y ~ N(theta_g, 1), theta_g ~ N(mu, tau^2).  logpdf selects theta_g with an
# unrolled compare-and-select so that theta stays in registers; the expressions are the oracle's.
HIER = r"""
constexpr int NGRP = EXTMCMC_P - 2;
struct Law { double th[NGRP]; double mu, tau, logtau; };
__device__ bool set_parameters(Law &L, const double *th) {
    const double tau = th[NGRP + 1];
    if (!(tau > 0.0) || isinf(tau)) return false;
    for (int g = 0; g < NGRP; ++g) L.th[g] = th[g];
    L.mu = th[NGRP];
    L.tau = tau;
    L.logtau = log(tau);
    return true;
}
__device__ double logpdf(const Law &L, const double *x) {
    double m = L.th[0];
#pragma unroll
    for (int g = 1; g < NGRP; ++g) m = x[1] == (double)g ? L.th[g] : m;
    const double r = x[0] - m;
    return -0.5 * 1.8378770664093453 - (r * r) / 2.0;
}
__device__ double logpdf_theta(const Law &L) {
    double s = 0.0;
    for (int g = 0; g < NGRP; ++g) {
        const double dv = L.th[g] - L.mu;
        s += -0.5 * 1.8378770664093453 - L.logtau - (dv * dv) / (2.0 * L.tau * L.tau);
    }
    return s;
}
"""

_HIER_GRADS = r"""
__device__ double logpdf_grad(const Law &L, const double *x, double *gr) {
    double m = L.th[0];
#pragma unroll
    for (int g = 1; g < NGRP; ++g) m = x[1] == (double)g ? L.th[g] : m;
    const double r = x[0] - m;
#pragma unroll
    for (int g = 0; g < NGRP; ++g)
        if (x[1] == (double)g) gr[g] += r;
    return -0.5 * 1.8378770664093453 - (r * r) / 2.0;
}
__device__ double logpdf_theta_grad(const Law &L, double *gr) {
    double s = 0.0;
    for (int g = 0; g < NGRP; ++g) {
        const double dv = L.th[g] - L.mu;
        s += -0.5 * 1.8378770664093453 - L.logtau - (dv * dv) / (2.0 * L.tau * L.tau);
        gr[g] += -dv / (L.tau * L.tau);
        gr[NGRP] += dv / (L.tau * L.tau);
        gr[NGRP + 1] += -1.0 / L.tau + (dv * dv) / (L.tau * L.tau * L.tau);
    }
    return s;
}
"""
HIER_HAND = HIER + _HIER_GRADS

HIER_FORWARD = r"""
constexpr int NGRP = EXTMCMC_P - 2;
template <class real> struct Law { real th[NGRP]; real mu, tau, logtau; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    const real tau = th[NGRP + 1];
    if (!(tau > 0.0) || isinf(tau)) return false;
    for (int g = 0; g < NGRP; ++g) L.th[g] = th[g];
    L.mu = th[NGRP];
    L.tau = tau;
    L.logtau = log(tau);
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    real m = L.th[0];
#pragma unroll
    for (int g = 1; g < NGRP; ++g) m = x[1] == (double)g ? L.th[g] : m;
    const real r = x[0] - m;
    return -0.5 * 1.8378770664093453 - (r * r) / 2.0;
}
template <class real> __device__ real logpdf_theta(const Law<real> &L) {
    real s = 0.0;
    for (int g = 0; g < NGRP; ++g) {
        const real dv = L.th[g] - L.mu;
        s += -0.5 * 1.8378770664093453 - L.logtau - (dv * dv) / (2.0 * L.tau * L.tau);
    }
    return s;
}
"""

# Poisson regression with a ridge penalty of unknown precision: theta = [beta_0..beta_{P-2}, log lambda],
# row = [x_1..x_{P-2}, y], D = P - 1; beta ~ N(0, 1 / lambda) iid up to its constant:
# logpdf_theta = (P - 1) / 2 log lambda - lambda / 2 |beta|^2.  log lambda appears in the term only.
RIDGE_POISSON = r"""
constexpr int NBETA = EXTMCMC_P - 1;
struct Law { double b[NBETA]; double loglam, lam; };
__device__ bool set_parameters(Law &L, const double *th) {
    for (int k = 0; k < NBETA; ++k) L.b[k] = th[k];
    L.loglam = th[NBETA];
    L.lam = exp(th[NBETA]);
    return true;
}
__device__ double lin(const Law &L, const double *x) {
    double e = L.b[0];
    for (int k = 1; k < NBETA; ++k) e += x[k - 1] * L.b[k];
    return e;
}
__device__ double logpdf(const Law &L, const double *x) {
    const double y = x[EXTMCMC_D - 1], e = lin(L, x);
    return y * e - exp(e);
}
__device__ double logpdf_grad(const Law &L, const double *x, double *g) {
    const double y = x[EXTMCMC_D - 1], e = lin(L, x), r = y - exp(e);
    g[0] += r;
    for (int k = 1; k < NBETA; ++k) g[k] += r * x[k - 1];
    return y * e - exp(e);
}
__device__ double logpdf_theta(const Law &L) {
    double s = 0.0;
    for (int k = 0; k < NBETA; ++k) s += L.b[k] * L.b[k];
    return 0.5 * NBETA * L.loglam - 0.5 * L.lam * s;
}
__device__ double logpdf_theta_grad(const Law &L, double *g) {
    double s = 0.0;
    for (int k = 0; k < NBETA; ++k) {
        s += L.b[k] * L.b[k];
        g[k] += -L.lam * L.b[k];
    }
    g[NBETA] += 0.5 * NBETA - 0.5 * L.lam * s;
    return 0.5 * NBETA * L.loglam - 0.5 * L.lam * s;
}
"""

RIDGE_POISSON_FORWARD = r"""
constexpr int NBETA = EXTMCMC_P - 1;
template <class real> struct Law { real b[NBETA]; real loglam, lam; };
template <class real> __device__ bool set_parameters(Law<real> &L, const real *th) {
    for (int k = 0; k < NBETA; ++k) L.b[k] = th[k];
    L.loglam = th[NBETA];
    L.lam = exp(th[NBETA]);
    return true;
}
template <class real> __device__ real logpdf(const Law<real> &L, const double *x) {
    real e = L.b[0];
    for (int k = 1; k < NBETA; ++k) e += x[k - 1] * L.b[k];
    return x[EXTMCMC_D - 1] * e - exp(e);
}
template <class real> __device__ real logpdf_theta(const Law<real> &L) {
    real s = 0.0;
    for (int k = 0; k < NBETA; ++k) s += L.b[k] * L.b[k];
    return 0.5 * NBETA * L.loglam - 0.5 * L.lam * s;
}
"""

# with the flag, each of these lacks a function the mode needs
NO_THETA_PLAIN = ul.POISSON_REG                                   # no logpdf_theta
NO_THETA_FORWARD = uf.POISSON_REG                                 # no template logpdf_theta
NO_THETA_GRAD = HIER + _HIER_GRADS.split("__device__ double logpdf_theta_grad")[0]   # hand mode: no logpdf_theta_grad


def hier_terms(theta, X, dtype=np.float64):
    """Per-row [N, C] and their gradients [P, N, C]; theta [P, C], X [N, 2] = [y, group]."""
    theta, X = np.asarray(theta, dtype), np.asarray(X, dtype)
    P = theta.shape[0]
    grp = X[:, 1].astype(int)
    r = X[:, :1] - theta[grp]
    t = -dtype(LOG2PI) / 2 - r * r / 2
    g = np.zeros((P,) + r.shape, dtype)
    g[grp, np.arange(len(grp))] = r
    return t, g


def hier_theta_term(theta, dtype=np.float64):
    """The theta term [C] and its gradient [P, C]."""
    theta = np.asarray(theta, dtype)
    Gn = theta.shape[0] - 2
    mu, tau = theta[Gn], theta[Gn + 1]
    dv = theta[:Gn] - mu
    v = (-dtype(LOG2PI) / 2 - np.log(tau) - dv * dv / (2 * tau * tau)).sum(axis=0)
    g = np.empty_like(theta)
    g[:Gn] = -dv / (tau * tau)
    g[Gn] = (dv / (tau * tau)).sum(axis=0)
    g[Gn + 1] = (-1 / tau + dv * dv / tau ** 3).sum(axis=0)
    return v, g


def ridge_terms(theta, X, dtype=np.float64):
    theta = np.asarray(theta, dtype)
    t, gb = ul.poisson_reg_terms(theta[:-1], X, dtype)
    return t, np.concatenate([gb, np.zeros((1,) + t.shape, dtype)])


def ridge_theta_term(theta, dtype=np.float64):
    theta = np.asarray(theta, dtype)
    b, loglam = theta[:-1], theta[-1]
    lam, nb, s = np.exp(loglam), b.shape[0], (b * b).sum(axis=0)
    v = nb / dtype(2) * loglam - lam / 2 * s
    return v, np.concatenate([-lam * b, (nb / dtype(2) - lam / 2 * s)[None]])


# name -> (plain / hand-gradient source, forward source, D(P), row terms, theta term)
LAWS = {
    "hier": (HIER_HAND, HIER_FORWARD, lambda P: 2, hier_terms, hier_theta_term),
    "ridge": (RIDGE_POISSON, RIDGE_POISSON_FORWARD, lambda P: P - 1, ridge_terms, ridge_theta_term),
}


def reference(name, theta, X, dtype=np.longdouble, chunk=16):
    """ll [C], gradient [P, C] and the sum of the gradient terms' magnitudes [P, C] (the scale of its
    rounding), in dtype."""
    _, _, _, terms, tterm = LAWS[name]
    Cn = theta.shape[1]
    ll, gr, gra = np.empty(Cn), np.empty(theta.shape), np.empty(theta.shape)
    lla = np.empty(Cn)
    for lo in range(0, Cn, chunk):
        th = theta[:, lo:lo + chunk]
        t, g = terms(th, X, dtype=dtype)
        v, gt = tterm(th, dtype=dtype)
        ll[lo:lo + chunk] = t.sum(axis=0) + v
        lla[lo:lo + chunk] = np.abs(t).sum(axis=0) + np.abs(v)
        gr[:, lo:lo + chunk] = g.sum(axis=1) + gt
        gra[:, lo:lo + chunk] = np.abs(g).sum(axis=1) + np.abs(gt)
    return ll, lla, gr, gra


def hier_data(N_per_group, seed=0, ragged=False, Gn=G):
    """Rows [N, 2] = [y, group], sorted by group, and the group index of every row."""
    rng = np.random.default_rng(seed)
    tg = rng.standard_normal(Gn)
    sizes = [N_per_group + (3 * g + 1 if ragged else 0) for g in range(Gn)]
    y = np.concatenate([tg[g] + rng.standard_normal(sizes[g]) for g in range(Gn)])
    grp = np.concatenate([np.full(sizes[g], g) for g in range(Gn)])
    return np.stack([y, grp.astype(np.float64)], axis=1), grp


def data(name, N, P, seed=0):
    if name == "hier":
        return hier_data(-(-N // (P - 2)), seed=seed, Gn=P - 2)[0][:N]
    rng = np.random.default_rng(seed)
    nx = P - 2
    X = np.empty((N, P - 1))
    X[:, :nx] = rng.standard_normal((N, nx)) / math.sqrt(max(nx, 1))
    beta = 0.5 * rng.standard_normal(P - 1)
    X[:, nx] = rng.poisson(np.exp(beta[0] + X[:, :nx] @ beta[1:]))
    return X


def theta(name, P, Cn, seed=1):
    """A state [P, C] in the law's domain."""
    rng = np.random.default_rng(seed)
    th = 0.3 * rng.standard_normal((P, Cn))
    if name == "hier":
        th[P - 1] = np.exp(0.2 * rng.standard_normal(Cn))
    return th
