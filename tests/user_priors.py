"""Sample user-defined priors (DevicePrior sources) shared by the CPU and GPU tests.

The restatements of built-in families use the association of step_device.cuh (log_prior_family,
prior_grad, prior_logpdf1): a sum over the coordinates in index order that starts at 0.0, each term the
built-in expression, so a restated prior gives the built-in prior's bits.  pp holds the family's
parameters in the order StandardPrior passes them."""

LOG2PI = "1.8378770664093454835606594728112"
LOGPI = "1.1447298858494001741434273513531"

# StandardPrior(Normal(m, sd)), pp = {m, sd}; value, hand-written gradient (prior_grad) and forward mode
NORMAL = f"""
__device__ double logprior(const double *th, const double *pp) {{
    double s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) {{
        const double z = (th[i] - pp[0]) / pp[1];
        s += -(z * z + {LOG2PI}) / 2.0 - log(pp[1]);
    }}
    return s;
}}
__device__ double logprior_grad(const double *th, const double *pp, double *g) {{
    for (int i = 0; i < EXTMCMC_PU; ++i) g[i] += -(th[i] - pp[0]) / (pp[1] * pp[1]);
    return logprior(th, pp);
}}
"""

NORMAL_FORWARD = f"""
template <class real> __device__ real logprior(const real *th, const double *pp) {{
    real s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) {{
        const real z = (th[i] - pp[0]) / pp[1];
        s += -(z * z + {LOG2PI}) / 2.0 - log(pp[1]);
    }}
    return s;
}}
"""

# StandardPrior(Gamma(k, scale)), pp = {k, scale}
GAMMA = """
__device__ double logprior(const double *th, const double *pp) {
    const double k = pp[0], sc = pp[1];
    double s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) {
        const double x = th[i];
        if (!(x > 0.0)) return -INFINITY;
        s += -lgamma(k) - k * log(sc) + (k - 1.0) * log(x) - x / sc;
    }
    return s;
}
"""

# StandardPrior(Uniform(a, b)), pp = {a, b}
UNIFORM = """
__device__ double logprior(const double *th, const double *pp) {
    const double a = pp[0], b = pp[1];
    double s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) {
        const double x = th[i];
        if (!(x >= a && x <= b)) return -INFINITY;
        s += -log(b - a);
    }
    return s;
}
"""

# StandardPrior(Beta(a, b)), pp = {a, b}
BETA = """
__device__ double logprior(const double *th, const double *pp) {
    const double a = pp[0], b = pp[1];
    const double lbeta = lgamma(a) + lgamma(b) - lgamma(a + b);
    double s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) {
        const double x = th[i];
        if (!(x > 0.0 && x < 1.0)) return -INFINITY;
        s += (a - 1.0) * log(x) + (b - 1.0) * log1p(-x) - lbeta;
    }
    return s;
}
"""

# StandardPrior(Cauchy(m, sc)), pp = {m, sc}
CAUCHY = f"""
__device__ double logprior(const double *th, const double *pp) {{
    double s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) {{
        const double z = (th[i] - pp[0]) / pp[1];
        s += -(log1p(z * z) + {LOGPI} + log(pp[1]));
    }}
    return s;
}}
"""

# ImproperPosPrior: -sum(log th)
IMPROPER_POS = """
__device__ double logprior(const double *th, const double *pp) {
    double s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) s += log(th[i]);
    return -s;
}
"""

# ProductPrior([Normal(m, sd), Gamma(k, sc)], [1, 1]) on two coordinates: pp = {m, sd, k, sc}.  The
# built-in sums the factors in order starting at 0.0: lp = (0 + normal) + gamma.
PRODUCT_NORMAL_GAMMA = f"""
__device__ double logprior(const double *th, const double *pp) {{
    double lp = 0.0;
    {{
        const double z = (th[0] - pp[0]) / pp[1];
        lp += 0.0 + (-(z * z + {LOG2PI}) / 2.0 - log(pp[1]));
    }}
    const double x = th[1], k = pp[2], sc = pp[3];
    if (!(x > 0.0)) return -INFINITY;
    lp += 0.0 + (-lgamma(k) - k * log(sc) + (k - 1.0) * log(x) - x / sc);
    return lp;
}}
"""

# Laplace(m, b) on each coordinate, pp = {m, b}: hand-written gradient (sign at the kink: 0)
LAPLACE = """
__device__ double logprior(const double *th, const double *pp) {
    double s = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) s += -fabs(th[i] - pp[0]) / pp[1] - log(2.0 * pp[1]);
    return s;
}
__device__ double logprior_grad(const double *th, const double *pp, double *g) {
    for (int i = 0; i < EXTMCMC_PU; ++i) {
        const double d = th[i] - pp[0];
        g[i] += d > 0.0 ? -1.0 / pp[1] : d < 0.0 ? 1.0 / pp[1] : 0.0;
    }
    return logprior(th, pp);
}
"""

# Student-t(nu) scaled by s on each coordinate, pp = {nu, s}; forward mode
STUDENT_T_FORWARD = """
template <class real> __device__ real logprior(const real *th, const double *pp) {
    const double nu = pp[0], s = pp[1];
    const double c = lgamma((nu + 1.0) / 2.0) - lgamma(nu / 2.0) - 0.5 * log(nu * 3.141592653589793) - log(s);
    real acc = 0.0;
    for (int i = 0; i < EXTMCMC_PU; ++i) {
        const real z = th[i] / s;
        acc += c - (nu + 1.0) / 2.0 * log1p(z * z / nu);
    }
    return acc;
}
"""

# does not compile: the log must name the undefined identifier
BAD = """
__device__ double logprior(const double *th, const double *pp) { return undefined_thing(th[0]); }
"""
