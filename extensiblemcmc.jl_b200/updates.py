"""Updates (src/updates.jl): transition kernel + coordinates + prior + adaptation."""
import numpy as np

from . import _abi
from .adaptation import NoAdaptation
from .priors import ImproperPrior
from .random_walk import RandomWalk
from .types import MCMCGradientBasedUpdate, MCMCParamUpdate


class RandomWalkUpdate(MCMCParamUpdate):
    """RandomWalkUpdate(rw, idx_of_global; prior=ImproperPrior(), adpt=NoAdaptation()) --
    src/updates.jl:163-183.  `coords` are 1-based indices into theta, as in the reference."""

    def __init__(self, rw, idx_of_global, prior=None, adpt=None):
        assert isinstance(rw, RandomWalk)
        self.rw = rw
        self.adpt = adpt if adpt is not None else NoAdaptation()
        self.coords = [int(i) for i in np.atleast_1d(idx_of_global)]
        self.invcoords = {c: i + 1 for i, c in enumerate(self.coords)}   # updates.jl:176-179
        self.prior = prior if prior is not None else ImproperPrior()
        if len(self.coords) != len(rw):
            raise ValueError("length(coords) must equal length(rw)")

    def to_abi(self, n_params):
        """-> (_abi.Update, keepalive) with 0-based coordinates."""
        coords = np.asarray(self.coords, dtype=np.int32) - 1
        if np.any(coords < 0) or np.any(coords >= n_params):
            raise ValueError("update coordinates out of range (1-based indices into theta)")
        step = np.ascontiguousarray(self.rw.abi_step(), dtype=np.float64)
        pos = np.ascontiguousarray(self.rw.pos, dtype=np.uint8)
        prior_kind, prior_params = self.prior.to_abi()
        prior_params = np.ascontiguousarray(prior_params, dtype=np.float64)
        u = _abi.Update()
        u.kernel = self.rw.abi_kernel
        u.n_coords = len(self.coords)
        u.coords = coords.ctypes.data_as(_abi.c_int32_p)
        u.step = step.ctypes.data_as(_abi.c_double_p)
        u.pos = pos.ctypes.data_as(_abi.c_uint8_p)
        u.prior = prior_kind
        u.n_prior_params = prior_params.size
        u.prior_params = prior_params.ctypes.data_as(_abi.c_double_p) if prior_params.size else None
        u.adapt = self.adpt.to_abi()
        return u, (coords, step, pos, prior_params)


def coords(updt):                                      # updates.jl:111
    return updt.coords


def invcoords(updt):                                   # updates.jl:113
    return updt.invcoords


class MALAUpdate(MCMCGradientBasedUpdate):
    """MALAUpdate(tau, idx_of_global; prior=ImproperPrior(), adpt=NoAdaptation()).

    An empty `#TODO` stub in the reference (src/updates.jl:216-218); only the hooks exist
    (MCMCGradientBasedUpdate src/types.jl:24, compute_gradients_and_momenta!
    src/updates.jl:129-133, the `grad ll` buffer src/workspaces.jl:417).  Build-defined
    semantics: theta° = theta + tau^2/2 * grad(ll + log prior)(theta) + tau * z, z ~ N(0, I),
    Metropolis-Hastings corrected with the same llr association and Exp(1) test as every other
    update (src/run.jl:268-281).  Priors: ImproperPrior, StandardPrior(Normal), and a DevicePrior
    with a gradient."""

    def __init__(self, tau, idx_of_global, prior=None, adpt=None):
        self.tau = float(tau)
        assert self.tau > 0.0
        self.adpt = adpt if adpt is not None else NoAdaptation()
        self.coords = [int(i) for i in np.atleast_1d(idx_of_global)]
        self.invcoords = {c: i + 1 for i, c in enumerate(self.coords)}
        self.prior = prior if prior is not None else ImproperPrior()

    def to_abi(self, n_params):
        coords = np.asarray(self.coords, dtype=np.int32) - 1
        if np.any(coords < 0) or np.any(coords >= n_params):
            raise ValueError("update coordinates out of range (1-based indices into theta)")
        step = np.array([self.tau], dtype=np.float64)
        prior_kind, prior_params = self.prior.to_abi()
        prior_params = np.ascontiguousarray(prior_params, dtype=np.float64)
        u = _abi.Update()
        u.kernel = _abi.KERNEL_MALA
        u.n_coords = len(self.coords)
        u.coords = coords.ctypes.data_as(_abi.c_int32_p)
        u.step = step.ctypes.data_as(_abi.c_double_p)
        u.pos = None
        u.prior = prior_kind
        u.n_prior_params = prior_params.size
        u.prior_params = prior_params.ctypes.data_as(_abi.c_double_p) if prior_params.size else None
        u.adapt = self.adpt.to_abi()
        return u, (coords, step, prior_params)


class HamiltonianMCUpdate(MCMCGradientBasedUpdate):    # updates.jl:220-222
    def to_abi(self, n_params):
        raise NotImplementedError("HamiltonianMCUpdate is not implemented (TODO stub in the reference)")
