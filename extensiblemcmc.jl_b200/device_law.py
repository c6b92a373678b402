"""DeviceLaw -- a user-defined target law on the device.

The reference lets users bring their own law: `set_parameters!(P, θ)` and `loglikelihood(P, obs)`
(docs/src/get_started/basic_use.md, src/example/gsn_target.jl).  Here the same two functions are
written in CUDA C++ and compiled at run time into the likelihood sweep (csrc/sweep_user.cuh,
csrc/user_law.cu; the contract is in include/extmcmc.h and INTEGRATION.md):

    struct Law { ... };                                              // per-chain constants
    __device__ bool   set_parameters(Law &L, const double *th);     // th[0..EXTMCMC_P-1]
    __device__ double logpdf(const Law &L, const double *x);        // x[0..EXTMCMC_D-1], one row
    __device__ double logpdf_grad(const Law &L, const double *x, double *g);   // gradient=True

With gradient="forward" the law is written once, generic over its scalar, and the library derives the
gradient in forward mode (dual numbers, csrc/dual.cuh; at most 16 parameters):

    template <class real> struct Law { real b[EXTMCMC_P]; };
    template <class real> __device__ bool set_parameters(Law<real> &L, const real *th);
    template <class real> __device__ real logpdf(const Law<real> &L, const double *x);

Up to 64 parameters in forward mode with chunk="auto" or a chunk width: the gradient is then ceil(P/K)
sweeps of K tangents each (ForwardDiff's chunk mode); the library picks K for "auto", and law.chunk
reports the width compiled.

With theta_term=True the law also defines a term of theta only, added once to its log-likelihood
(sum over rows of logpdf, plus logpdf_theta): the hierarchical p(theta_g | mu, tau) of a multilevel model,
a shrinkage penalty, any term the reference's loglikelihood adds that no row carries:

    __device__ double logpdf_theta(const Law &L);
    __device__ double logpdf_theta_grad(const Law &L, double *g);                  // gradient=True
    template <class real> __device__ real logpdf_theta(const Law<real> &L);        // gradient="forward"

With theta_only (1-based coordinates, like the updates'), the law also declares which coordinates its
rows do not read: logpdf and logpdf_grad do not depend on them, only logpdf_theta does.  A random-walk
update of those coordinates alone (the mu and tau of a hierarchical model) then runs without a
likelihood sweep, and a MALA update after it reuses the rows' part of its gradient.  The declaration is
not verified: run the same seed with EXTMCMC_DATA_CACHE=0 and compare (a true one gives the same bits).

Data: dict(P=DeviceLaw(source, n_params, obs_dim), obs=rows [N, obs_dim]); responses and
covariates are columns of the rows.  The constructor compiles the law for sm_100a (no device
needed) and raises ValueError with the compiler's log when it does not compile.
"""
import ctypes as C

from . import _abi


class DeviceLaw:
    def __init__(self, source, n_params, obs_dim=1, gradient=False, chunk=None, theta_term=False, theta_only=None):
        """gradient: False (none), True (the source defines logpdf_grad) or "forward".
        chunk (forward mode only): None (unchunked, at most 16 parameters), "auto" (the library's width)
        or a chunk width; the library checks the width against n_params.
        theta_term: True when the source defines logpdf_theta (and logpdf_theta_grad with gradient=True).
        theta_only: None, or the 1-based coordinates the rows do not read (needs theta_term=True)."""
        if isinstance(gradient, str) and gradient == "forward":
            self._with_grad = _abi.USER_GRAD_FORWARD
        elif isinstance(gradient, (bool, int)) and gradient in (False, True):
            self._with_grad = _abi.USER_GRAD_HAND if gradient else _abi.USER_GRAD_NONE
        else:
            raise ValueError(f"gradient must be False, True or 'forward', not {gradient!r}")
        if chunk is not None and self._with_grad != _abi.USER_GRAD_FORWARD:
            raise ValueError(f"chunk needs gradient='forward', not gradient={gradient!r}")
        if chunk is None or (isinstance(chunk, str) and chunk == "auto"):
            self._chunk_arg = None if chunk is None else 0
        elif isinstance(chunk, int) and not isinstance(chunk, bool) and chunk >= 1:
            self._chunk_arg = chunk
        else:
            raise ValueError(f"chunk must be None, 'auto' or a positive width, not {chunk!r}")
        if not isinstance(theta_term, bool):
            raise ValueError(f"theta_term must be True or False, not {theta_term!r}")
        self.theta_term = theta_term
        self.theta_only = self._theta_only(theta_only, int(n_params), theta_term)
        self.source = str(source)
        self._n_params = int(n_params)
        self._obs_dim = int(obs_dim)
        self.gradient = "forward" if self._with_grad == _abi.USER_GRAD_FORWARD else bool(gradient)
        self.chunk = None                            # forward mode: the chunk width compiled
        lib = _abi.load()
        buf = C.create_string_buffer(1 << 16)
        if self.theta_only is not None:
            used = C.c_int32(-1)
            rc = lib.extmcmc_user_law_check_theta_only(self.source.encode(), self._n_params, self._obs_dim,
                                                       self._with_grad, self._ex_chunk(), _abi.USER_THETA_TERM,
                                                       self._theta_only_mask(), C.byref(used), buf, len(buf))
            if rc == _abi.EINVAL and used.value == -1:   # the arguments were refused before compiling
                raise ValueError(buf.value.decode(errors="replace"))
            if self._with_grad == _abi.USER_GRAD_FORWARD:
                self.chunk = used.value
        elif theta_term:
            used = C.c_int32(-1)
            rc = lib.extmcmc_user_law_check_ex(self.source.encode(), self._n_params, self._obs_dim, self._with_grad,
                                               self._ex_chunk(), _abi.USER_THETA_TERM, C.byref(used), buf, len(buf))
            if rc == _abi.EINVAL and used.value == -1:   # the arguments were refused before compiling
                raise ValueError(buf.value.decode(errors="replace"))
            if self._with_grad == _abi.USER_GRAD_FORWARD:
                self.chunk = used.value
        elif self._chunk_arg is None:
            rc = lib.extmcmc_user_law_check(self.source.encode(), self._n_params, self._obs_dim,
                                            self._with_grad, buf, len(buf))
            if rc == _abi.OK and self._with_grad == _abi.USER_GRAD_FORWARD:
                self.chunk = self._n_params
        else:
            used = C.c_int32(0)
            rc = lib.extmcmc_user_law_check_chunked(self.source.encode(), self._n_params, self._obs_dim,
                                                    self._chunk_arg, C.byref(used), buf, len(buf))
            if rc == _abi.EINVAL and used.value == 0:   # the width was refused before compiling
                raise ValueError(buf.value.decode(errors="replace"))
            self.chunk = used.value
        self.log = buf.value.decode(errors="replace")   # NVRTC + ptxas log (registers, spill bytes)
        if rc == _abi.EINVAL:
            raise ValueError("the device law does not compile:\n" + self.log)
        if rc != _abi.OK:
            raise _abi.ExtMCMCError(rc, self.log or lib.extmcmc_last_error(None).decode())

    @staticmethod
    def _theta_only(theta_only, n_params, theta_term):
        """theta_only as a sorted tuple of 1-based coordinates, or None"""
        if theta_only is None:
            return None
        if isinstance(theta_only, (str, bytes)):
            raise ValueError(f"theta_only must be None or an iterable of 1-based coordinates, not {theta_only!r}")
        try:
            coords = list(theta_only)
        except TypeError:
            raise ValueError(f"theta_only must be None or an iterable of 1-based coordinates, not {theta_only!r}")
        if not theta_term:
            raise ValueError("theta_only needs theta_term=True: only logpdf_theta may read those coordinates")
        if not coords:
            raise ValueError("theta_only declares no coordinate (use None)")
        for k in coords:
            if isinstance(k, bool) or not isinstance(k, int):
                raise ValueError(f"theta_only coordinates must be integers, not {k!r}")
            if not 1 <= k <= n_params:
                raise ValueError(f"theta_only coordinate {k} is outside 1..{n_params}")
        if len(set(coords)) != len(coords):
            raise ValueError(f"theta_only lists a coordinate twice: {coords}")
        return tuple(sorted(coords))

    def _theta_only_mask(self):
        """bit k = 0-based coordinate k"""
        return sum(1 << (k - 1) for k in self.theta_only)

    def _ex_chunk(self):
        """chunk of the _ex entry points: None in forward mode is the unchunked width n_params"""
        if self._chunk_arg is not None:
            return self._chunk_arg
        return self._n_params if self._with_grad == _abi.USER_GRAD_FORWARD else 0

    def abi_law(self):
        return _abi.LAW_USER

    @property
    def n_params(self):
        return self._n_params

    @property
    def obs_dim(self):
        return self._obs_dim

    def abi_y(self, data=None):
        return None                                  # responses are columns of the rows

    def abi_attach(self, lib, handle):
        """Compiles (cached) and installs the law on a freshly created library handle."""
        if self.theta_only is not None:
            return lib.extmcmc_set_user_law_theta_only(handle, self.source.encode(), self._with_grad, self._ex_chunk(),
                                                       _abi.USER_THETA_TERM, self._theta_only_mask())
        if self.theta_term:
            return lib.extmcmc_set_user_law_ex(handle, self.source.encode(), self._with_grad, self._ex_chunk(),
                                               _abi.USER_THETA_TERM)
        if self._chunk_arg is not None:
            return lib.extmcmc_set_user_law_chunked(handle, self.source.encode(), self._chunk_arg)
        return lib.extmcmc_set_user_law(handle, self.source.encode(), self._with_grad)
