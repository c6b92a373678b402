"""Priors (src/priors.jl).  Evaluated on the device on the update's own coordinates only
(src/run.jl:374-385, src/updates.jl:104).  Arbitrary `dist` objects cannot cross the C ABI:
the enumerated families below are supported, anything else raises at workspace creation
(the reference's convention for a missing method is error("... not implemented")).  A prior of any
other form is written as CUDA C++ and compiled at run time: DevicePrior."""
import ctypes as C

import numpy as np

from . import _abi


class Prior:                                          # priors.jl:4
    def to_abi(self):
        raise NotImplementedError(f"logpdf not implemented for prior {type(self).__name__} on the GPU path")


class ImproperPrior(Prior):                           # priors.jl:18-19
    def to_abi(self):
        return _abi.PRIOR_IMPROPER, np.zeros(0)


class ImproperPosPrior(Prior):                        # priors.jl:25-26
    def to_abi(self):
        return _abi.PRIOR_IMPROPER_POS, np.zeros(0)


class Normal:
    """Stand-in for Distributions.Normal(mu, sigma) inside StandardPrior."""
    def __init__(self, mu=0.0, sigma=1.0):
        self.mu, self.sigma = float(mu), float(sigma)


class Gamma:
    """Stand-in for Distributions.Gamma(shape, scale)."""
    def __init__(self, shape=1.0, scale=1.0):
        self.shape, self.scale = float(shape), float(scale)


class Uniform:
    """Stand-in for Distributions.Uniform(a, b)."""
    def __init__(self, a=0.0, b=1.0):
        self.a, self.b = float(a), float(b)


class Exponential:
    """Stand-in for Distributions.Exponential(scale)."""
    def __init__(self, scale=1.0):
        self.scale = float(scale)


class InverseGamma:
    """Stand-in for Distributions.InverseGamma(shape, scale)."""
    def __init__(self, shape=1.0, scale=1.0):
        self.shape, self.scale = float(shape), float(scale)


class Beta:
    """Stand-in for Distributions.Beta(alpha, beta)."""
    def __init__(self, alpha=1.0, beta=1.0):
        self.alpha, self.beta = float(alpha), float(beta)


class LogNormal:
    """Stand-in for Distributions.LogNormal(mu, sigma)."""
    def __init__(self, mu=0.0, sigma=1.0):
        self.mu, self.sigma = float(mu), float(sigma)


class Cauchy:
    """Stand-in for Distributions.Cauchy(mu, sigma)."""
    def __init__(self, mu=0.0, sigma=1.0):
        self.mu, self.sigma = float(mu), float(sigma)


class MvNormal:
    """Stand-in for Distributions.MvNormal(mu, Sigma): a joint prior over the whole coordinate
    block of an update (priors.jl:35-39 wraps any Distributions object).  The host factorises
    Sigma = L L'; the device whitens with L, as PDMats does."""
    def __init__(self, mu, Sigma):
        self.mu = np.atleast_1d(np.asarray(mu, dtype=np.float64)).copy()
        self.Sigma = np.atleast_2d(np.asarray(Sigma, dtype=np.float64)).copy()
        n = self.mu.size
        if self.Sigma.shape != (n, n):
            raise ValueError("MvNormal: Sigma must be length(mu) x length(mu)")
        self.L = np.linalg.cholesky(self.Sigma)       # raises if not positive definite (PosDefException)


class StandardPrior(Prior):                           # priors.jl:35-39
    """StandardPrior(dist): a univariate `dist` is applied independently to each coordinate of
    the update (an iid product); an MvNormal covers the update's coordinate block jointly."""
    def __init__(self, dist):
        self.dist = dist

    def to_abi(self):
        d = self.dist
        if isinstance(d, Normal):
            return _abi.PRIOR_NORMAL, np.array([d.mu, d.sigma])
        if isinstance(d, Gamma):
            return _abi.PRIOR_GAMMA, np.array([d.shape, d.scale])
        if isinstance(d, Uniform):
            return _abi.PRIOR_UNIFORM, np.array([d.a, d.b])
        if isinstance(d, Exponential):
            return _abi.PRIOR_EXPONENTIAL, np.array([d.scale])
        if isinstance(d, InverseGamma):
            return _abi.PRIOR_INV_GAMMA, np.array([d.shape, d.scale])
        if isinstance(d, Beta):
            return _abi.PRIOR_BETA, np.array([d.alpha, d.beta])
        if isinstance(d, LogNormal):
            return _abi.PRIOR_LOGNORMAL, np.array([d.mu, d.sigma])
        if isinstance(d, Cauchy):
            return _abi.PRIOR_CAUCHY, np.array([d.mu, d.sigma])
        if isinstance(d, MvNormal):
            # {mu[n], L[n*n] column-major}
            return _abi.PRIOR_MVNORMAL, np.concatenate([d.mu, np.ascontiguousarray(d.L.T).ravel()])
        raise NotImplementedError(
            f"StandardPrior({type(d).__name__}) is not implemented on the GPU path (supported: Normal, "
            "Gamma, Uniform, Exponential, InverseGamma, Beta, LogNormal, Cauchy, MvNormal)")


class ProductPrior(Prior):                            # priors.jl:60-88
    """ProductPrior(dists, dims): factor k applies to the next dims[k] coordinates of the update
    (consecutive index groups, priors.jl:66-78).  Each factor is an ImproperPrior /
    ImproperPosPrior or one of the distribution stand-ins above (iid within its group)."""

    def __init__(self, dists, dims):
        self.dists, self.dims = tuple(dists), tuple(int(d) for d in dims)
        assert len(self.dists) == len(self.dims)

    def to_abi(self):
        out = [float(len(self.dists))]
        for dist, dim in zip(self.dists, self.dims):
            pr = dist if isinstance(dist, Prior) else StandardPrior(dist)
            kind, pp = pr.to_abi()
            if kind in (_abi.PRIOR_PRODUCT, _abi.PRIOR_MVNORMAL, _abi.PRIOR_USER):
                raise NotImplementedError("ProductPrior factors must be iid families on the GPU path")
            pp = list(pp) + [0.0, 0.0]
            out += [float(kind), float(dim), pp[0], pp[1]]
        return _abi.PRIOR_PRODUCT, np.array(out)


class DevicePrior(Prior):
    """A user-defined prior on the device: the reference's open Prior type (a subtype with
    logpdf(prior, th), priors.jl:4-39) written as CUDA C++ over the update's own EXTMCMC_PU coordinates
    and compiled at run time (csrc/prior_user.cuh; the contract is in include/extmcmc.h and INTEGRATION.md):

        __device__ double logprior(const double *th, const double *pp);            // -INFINITY off the support
        __device__ double logprior_grad(const double *th, const double *pp, double *g);   // gradient=True
        template <class real> __device__ real logprior(const real *th, const double *pp); // gradient="forward"

    pp are `params`, passed at run time (new hyperparameters need no recompilation).  Usable as the
    prior= of RandomWalkUpdate (the proposal is redrawn while logprior is -INFINITY) and, with a
    gradient, of MALAUpdate.  The constructor compiles the source for sm_100a at n_coords coordinates
    (default 1; the workspace compiles it again at its update's p_u) and raises ValueError with the
    compiler's log when it does not compile."""

    def __init__(self, source, gradient=False, params=(), n_coords=1):
        if isinstance(gradient, str) and gradient == "forward":
            self._with_grad = _abi.USER_GRAD_FORWARD
        elif isinstance(gradient, (bool, int)) and gradient in (False, True):
            self._with_grad = _abi.USER_GRAD_HAND if gradient else _abi.USER_GRAD_NONE
        else:
            raise ValueError(f"gradient must be False, True or 'forward', not {gradient!r}")
        self.source = str(source)
        self.gradient = "forward" if self._with_grad == _abi.USER_GRAD_FORWARD else bool(gradient)
        self.params = np.ascontiguousarray(np.atleast_1d(np.asarray(params, dtype=np.float64)))
        self.log = self.check(int(n_coords))

    def check(self, n_coords):
        """Compiles the prior's kernels for n_coords coordinates; returns the NVRTC + ptxas log
        (registers, spill bytes).  ValueError when the source does not compile."""
        lib = _abi.load()
        buf = C.create_string_buffer(1 << 16)
        rc = lib.extmcmc_user_prior_check(self.source.encode(), n_coords, self._with_grad, buf, len(buf))
        log = buf.value.decode(errors="replace")
        if rc == _abi.EINVAL:
            raise ValueError("the device prior does not compile:\n" + log)
        if rc != _abi.OK:
            raise _abi.ExtMCMCError(rc, log or lib.extmcmc_last_error(None).decode())
        return log

    def to_abi(self):
        return _abi.PRIOR_USER, self.params

    def abi_attach(self, lib, handle, u):
        """Compiles (cached) and installs the prior of update u (0-based), after extmcmc_set_update."""
        return lib.extmcmc_set_user_prior(handle, u, self.source.encode(), self._with_grad)
