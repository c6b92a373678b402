"""Device-resident workspaces of the CUDA backend.

Replaces, behind the reference's own backend seam, `init_global_workspace(::Backend, ...)`
(src/workspaces.jl:38-47,215-234) and `create_workspace(::Backend, updt, global_ws, M)`
(src/workspaces.jl:280-287,460-473).  The chain state, step sizes, counters, running
moments and a history ring live on the GPU (csrc/dev_state.cuh); the host objects below
own the library handle and host mirrors of the histories, filled at block boundaries,
and expose the reference's accessor names:

    reference (Julia)            here (Python)
    state(ws)                    state(ws)
    state(ws, step)              state(ws, step)
    state°(ws, step)             state_prop(ws, step)
    ll(ws) / ll°(ws)             ll(ws) / ll_prop(ws)
    ll(ws, i) / ll°(ws, i)       ll(ws, i) / ll_prop(ws, i)
    accepted(ws, i)              accepted(ws, i)
    estim_mean / estim_cov       estim_mean / estim_cov
    num_mcmc_steps / num_updt    num_mcmc_steps / num_updt

Every per-chain quantity carries a trailing chain axis of length n_chains (the reference
has exactly one chain; with n_chains = 1 squeeze the last axis to get its shapes).
Iteration and update indices are 1-based as in the reference.
"""
import ctypes as C

import numpy as np

from . import _abi
from .types import GenericMCMCBackend, GlobalWorkspace, LocalWorkspace, MCMCBackend


class CUDAMCMCBackend(MCMCBackend):
    """MCMC(updates; backend=CUDAMCMCBackend(n_chains=4096, ...)) selects the B200 path.

    n_chains       chains resident on this rank (independent replicas of the sampler)
    device         CUDA ordinal
    seed           Philox key; chain c uses the substream of global id chain_offset + c
    block_len      schedule elements shipped to the device per launch (one CUDA graph)
    history        "full": every (iteration, update) row is copied back (reference
                   behaviour); "none": histories stay on the device ring only
    stats_mode     0 mean + covariance (reference), 1 mean + variances, 2 off
                   (default: 0 for p <= 16 parameters, 1 above)
    shard_mode     "chains" (default) or "obs" (observations sharded over ranks, NCCL)
    rank/world_size/chain_offset  one process per GPU; see parallel.py
    """

    def __init__(self, n_chains=1, device=0, seed=0, block_len=128, history="full",
                 stats_mode=None, use_graphs=True, instrument=False, sweep_variant=0,
                 shard_mode="chains", rank=0, world_size=1, chain_offset=0, roll_window=100,
                 comm_id=None, p2p_allgather=None):
        assert history in ("full", "none")
        assert shard_mode in ("chains", "obs")
        self.n_chains = int(n_chains)
        self.device = int(device)
        self.seed = int(seed)
        self.block_len = int(block_len)
        self.history = history
        self.stats_mode = None if stats_mode is None else int(stats_mode)   # None: 0 if p <= 16 else 1
        self.use_graphs = bool(use_graphs)
        self.instrument = bool(instrument)
        self.sweep_variant = int(sweep_variant)
        self.shard_mode = shard_mode
        self.rank, self.world_size, self.chain_offset = int(rank), int(world_size), int(chain_offset)
        self.roll_window = int(roll_window)
        self.comm_id = comm_id
        # callable bytes -> [bytes of every rank, rank order]; enables the library's own NVLink
        # peer exchange of the per-chain sums instead of ncclAllReduce (shard_mode="obs")
        self.p2p_allgather = p2p_allgather
        self.runs_started = 0


def _run_seed(seed, run):
    """Philox key of the run-th run of a backend: the seed itself for run 0, a SplitMix64 mix after."""
    if run == 0:
        return seed & 0xFFFFFFFFFFFFFFFF
    z = (seed + run * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)


class _GlobalSub:
    """Counterpart of StandardGlobalSubworkspace (src/workspaces.jl:157-180)."""

    def __init__(self, M, NU, p, C, data, keep):
        self.data = data
        self.state = None                                     # [p, C], refreshed at block ends
        if keep:
            # rows are written block by block as they arrive from the device; rows of
            # schedule elements that never ran are NaN-filled at the end of run_ (the
            # reference leaves them `undef`, src/workspaces.jl:171)
            self.state_history = np.empty((M, NU, p, C))
            self.state_proposal_history = np.empty((M, NU, p, C))
        else:
            self.state_history = self.state_proposal_history = None
        self.stats = None


class CUDAGlobalWorkspace(GlobalWorkspace):
    def __init__(self, backend, num_mcmc_steps, updates, data, theta_init):
        lib = _abi.load()
        law = data["P"] if isinstance(data, dict) else data.P
        obs = data["obs"] if isinstance(data, dict) else data.obs
        if not hasattr(law, "abi_law"):
            raise NotImplementedError(
                f"target law {type(law).__name__} is not implemented on the GPU path "
                "(write it as a DeviceLaw: set_parameters / logpdf in CUDA C++)")
        self.backend = backend
        self.lib = lib
        self.M = int(num_mcmc_steps)
        self.NU = len(updates)
        self.p = law.n_params
        self.C = backend.n_chains
        self.P = law
        theta_init = np.asarray(theta_init, dtype=np.float64)
        if theta_init.ndim == 1:                              # one vector, replicated to all chains
            theta_init = np.repeat(theta_init[:, None], self.C, axis=1)
        if theta_init.shape != (self.p, self.C):
            raise ValueError(f"theta_init must have shape ({self.p},) or ({self.p}, {self.C})")
        self.theta_init = np.ascontiguousarray(theta_init)

        cfg = _abi.Config()
        cfg.abi_version = _abi.ABI_VERSION
        cfg.device = backend.device
        cfg.n_chains = self.C
        cfg.chain_offset = backend.chain_offset
        cfg.n_params = self.p
        cfg.n_updates = self.NU
        cfg.law = law.abi_law()
        cfg.obs_dim = law.obs_dim
        # the reference advances a global RNG from run to run; a counter RNG restarts, so every
        # further run of the same backend gets its own key (run 0 keeps the user's seed)
        cfg.seed = _run_seed(backend.seed, backend.runs_started)
        backend.runs_started += 1
        cfg.shard_mode = _abi.SHARD_OBS if backend.shard_mode == "obs" else _abi.SHARD_CHAINS
        cfg.rank, cfg.world_size = backend.rank, backend.world_size
        self.block_len = max(1, backend.block_len)
        cfg.history_window = 2 * self.block_len
        cfg.roll_window = backend.roll_window
        cfg.use_graphs = 1 if backend.use_graphs else 0
        cfg.instrument = 1 if backend.instrument else 0
        cfg.sweep_variant = backend.sweep_variant
        cfg.stats_mode = backend.stats_mode if backend.stats_mode is not None else (0 if self.p <= 16 else 1)
        backend.stats_mode = cfg.stats_mode
        self.cfg = cfg
        self.handle = _abi.Handle()
        rc = lib.extmcmc_create(C.byref(cfg), C.byref(self.handle))
        if rc != _abi.OK:
            msg = lib.extmcmc_last_error(None)
            raise _abi.ExtMCMCError(rc, msg.decode() if msg else "")
        try:
            if hasattr(law, "abi_attach"):                      # DeviceLaw: compile and install the law
                self._ck(law.abi_attach(lib, self.handle))
            if backend.comm_id is not None:
                ida = np.frombuffer(bytes(backend.comm_id), dtype=np.uint8).copy()
                self._ck(lib.extmcmc_comm_init(self.handle, ida.ctypes.data_as(_abi.c_uint8_p)))
            if backend.p2p_allgather is not None:
                mine = (C.c_uint8 * 64)()
                self._ck(lib.extmcmc_p2p_export(self.handle, mine))
                allh = backend.p2p_allgather(bytes(mine))
                buf = np.frombuffer(b"".join(allh), dtype=np.uint8).copy()
                assert buf.size == 64 * backend.world_size
                self._ck(lib.extmcmc_p2p_import(self.handle, buf.ctypes.data_as(_abi.c_uint8_p)))
            self._keep = []
            self._kernels = []
            for i, updt in enumerate(updates):
                if not hasattr(updt, "to_abi"):
                    raise NotImplementedError(f"update {type(updt).__name__} is not implemented on the GPU path")
                u, keep = updt.to_abi(self.p)
                self._keep.append(keep)
                self._kernels.append(u.kernel)
                self._ck(lib.extmcmc_set_update(self.handle, i, C.byref(u)))
                cb = getattr(getattr(updt, "adpt", None), "lambda_callback", lambda: None)()
                if cb is not None:                              # HaarioTypeAdaptation(...; f = ...)
                    self._keep.append(cb)
                    self._ck(lib.extmcmc_set_lambda_fn(self.handle, i, cb, None))
            if isinstance(obs, DeviceGeneratedObs):
                self._ck(lib.extmcmc_generate_obs_normal(self.handle, obs.first, obs.n, obs.mean, obs.sd, obs.seed))
                self.n_obs = obs.n
            else:
                obs = np.ascontiguousarray(np.asarray(obs, dtype=np.float64))
                if obs.ndim == 1:
                    obs = obs[:, None] if law.obs_dim == 1 else obs[None, :]
                if obs.shape[1] != law.obs_dim:
                    raise ValueError("observations must have shape (n_obs, obs_dim)")
                self.n_obs = obs.shape[0]
                y = law.abi_y(data) if hasattr(law, "abi_y") else None
                if y is not None and y.shape[0] != self.n_obs:
                    raise ValueError("one group index / response per observation is required")
                self._ck(lib.extmcmc_upload_obs(self.handle, _abi.dptr(obs), self.n_obs, law.obs_dim, _abi.dptr(y)))
            self._ck(lib.extmcmc_set_state(self.handle, _abi.dptr(self.theta_init)))
        except Exception:
            lib.extmcmc_destroy(self.handle)
            self.handle = None
            raise
        self.keep_history = backend.history == "full"
        self.sub_ws = _GlobalSub(self.M, self.NU, self.p, self.C, data, self.keep_history)
        self.sub_ws.state = self.theta_init.copy()
        if self.keep_history:
            # one contiguous array per quantity, [M][NU][C]; the local workspaces hold views
            self.ll_all = np.zeros((self.M, self.NU, self.C))            # workspaces.jl:426 (zeros)
            self.llp_all = np.zeros((self.M, self.NU, self.C))
            self.acc_all = np.zeros((self.M, self.NU, self.C), dtype=np.uint8)
            self.executed = np.zeros((self.M, self.NU), dtype=bool)
        self._n_local = 0
        self.local_wss = None

    # ---- plumbing ----------------------------------------------------------------
    def _ck(self, rc):
        return _abi.check(self.handle, rc)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.extmcmc_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._ck(self.lib.extmcmc_sync(self.handle))

    def refresh_state(self):
        th = np.empty((self.p, self.C))
        ll = np.empty(self.C)
        self._ck(self.lib.extmcmc_get_state(self.handle, _abi.dptr(th), _abi.dptr(ll)))
        self.sub_ws.state = th
        return th, ll

    def stats(self):
        """GenericChainStats per chain: mean [p, C], cov [p, p, C], rolling_ar [NU, C],
        n_accept / n_prop [NU, C]."""
        p, Cn, NU = self.p, self.C, self.NU
        mode = self.backend.stats_mode
        mean = np.empty((p, Cn)) if mode != 2 else None
        cov = (np.empty((p * p, Cn)) if mode == 0 else np.empty((p, Cn))) if mode != 2 else None
        ra = np.empty((NU, Cn))
        na = np.empty((NU, Cn), dtype=np.int64)
        npr = np.empty((NU, Cn), dtype=np.int64)
        self._ck(self.lib.extmcmc_get_stats(
            self.handle, _abi.dptr(mean), _abi.dptr(cov), _abi.dptr(ra),
            na.ctypes.data_as(_abi.c_int64_p), npr.ctypes.data_as(_abi.c_int64_p)))
        if mode == 0:
            cov = cov.reshape(p, p, Cn).transpose(1, 0, 2)      # column-major (a + b p) -> [a, b, C]
        return dict(mean=mean, cov=cov, rolling_ar=ra, n_accept=na, n_prop=npr)

    def eps(self, u):
        """Current per-chain step-size state of update u (1-based): eps [p_u, C] for a uniform
        walk, Sigma_B [p_u^2, C] (column-major) for a Gaussian mixture walk."""
        n = len(self._keep[u - 1][0])
        k = self._kernels[u - 1]
        rows = n * n if k == _abi.KERNEL_RW_GAUSS_MIX else (1 if k == _abi.KERNEL_MALA else n)
        out = np.empty((rows, self.C))
        self._ck(self.lib.extmcmc_get_eps(self.handle, u - 1, _abi.dptr(out)))
        return out

    def adapt_state(self, u):
        """HaarioTypeAdaptation mean [p_u, C] and cov [p_u^2, C] of update u (1-based)."""
        n = len(self._keep[u - 1][0])
        mean, cov = np.empty((n, self.C)), np.empty((n * n, self.C))
        self._ck(self.lib.extmcmc_get_adapt_state(self.handle, u - 1, _abi.dptr(mean), _abi.dptr(cov)))
        return mean, cov

    def checkpoint(self):
        """Everything a continued run depends on (state, step sizes, counters, moments, bookkeeping) as
        bytes; restore() puts it into a workspace created with the same configuration."""
        n = C.c_int64()
        self._ck(self.lib.extmcmc_checkpoint_size(self.handle, C.byref(n)))
        buf = (C.c_uint8 * n.value)()
        self._ck(self.lib.extmcmc_checkpoint_save(self.handle, buf, n.value))
        return bytes(buf)

    def restore(self, blob):
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        self._ck(self.lib.extmcmc_checkpoint_load(self.handle, buf, len(blob)))
        self.refresh_state()

    def eval_loglik(self):
        out = np.empty(self.C)
        self._ck(self.lib.extmcmc_eval_loglik(self.handle, _abi.dptr(out)))
        return out

    def eval_grad(self):
        """(ll [C], d ll / d theta [p, C]) at the current state (laws with a device gradient)."""
        ll, g = np.empty(self.C), np.empty((self.p, self.C))
        self._ck(self.lib.extmcmc_eval_grad(self.handle, _abi.dptr(ll), _abi.dptr(g)))
        return ll, g


class DeviceGeneratedObs:
    """data.obs placeholder: x_i ~ N(mean, sd^2) generated on the device from
    Philox(seed), global indices [first, first + n) -- BASELINE cfg 5 (N = 1e9)."""

    def __init__(self, n, mean, sd, seed, first=0):
        self.n, self.mean, self.sd, self.seed, self.first = int(n), float(mean), float(sd), int(seed), int(first)


class _LocalSub:
    """Counterpart of StandardLocalSubworkspace (src/workspaces.jl:413-431)."""

    def __init__(self, p_u, C, ll_hist_view):
        self.state = np.full((p_u, C), np.nan)
        self.ll = np.full((1, C), -np.inf)                      # workspaces.jl:425
        self.ll_history = ll_hist_view                          # [M, 1, C] view (workspaces.jl:426)


class CUDALocalWorkspace(LocalWorkspace):
    """Counterpart of GenericLocalWorkspace (src/workspaces.jl:453-458)."""

    def __init__(self, updt, global_ws, M):
        p_u = len(updt.coords)
        keep = global_ws.keep_history
        j = global_ws._n_local
        global_ws._n_local += 1
        self.sub_ws = _LocalSub(p_u, global_ws.C, global_ws.ll_all[:, j:j + 1] if keep else None)
        self.sub_ws_prop = _LocalSub(p_u, global_ws.C, global_ws.llp_all[:, j:j + 1] if keep else None)  # sub_ws°
        idx = np.asarray(updt.coords) - 1
        self.sub_ws.state[:] = global_ws.theta_init[idx]
        self.sub_ws_prop.state[:] = global_ws.theta_init[idx]
        self.acceptance_history = global_ws.acc_all[:, j].view(np.bool_) if keep else None
        self.updt_name = type(updt).__name__


# ---- backend dispatch (the reference's seam) -------------------------------------
def init_global_workspace(backend, num_mcmc_steps, updates, data, theta_init, **kwargs):
    if isinstance(backend, CUDAMCMCBackend):
        return CUDAGlobalWorkspace(backend, num_mcmc_steps, updates, data, theta_init)
    if isinstance(backend, GenericMCMCBackend):
        raise NotImplementedError(
            "GenericMCMCBackend is the reference's CPU sampler; this package provides only "
            "the B200 path (backend=CUDAMCMCBackend(...)) and has no CPU fallback")
    # src/workspaces.jl:46
    raise NotImplementedError(f"init_global_workspace not implemented for backend {type(backend).__name__}")


def create_workspace(backend, updt, global_ws, num_mcmc_steps):
    if isinstance(backend, CUDAMCMCBackend):
        return CUDALocalWorkspace(updt, global_ws, num_mcmc_steps)
    raise NotImplementedError(f"create_workspace not implemented for backend {type(backend).__name__}")


def create_workspaces(backend, mcmc):                           # src/workspaces.jl:362-371
    wss = [create_workspace(backend, mcmc.updates[i], mcmc.workspace, mcmc.schedule.num_mcmc_steps)
           for i in range(mcmc.schedule.num_updates)]
    mcmc.workspace.local_wss = wss
    return wss


# ---- accessors (src/workspaces.jl:91-136, 294-385) ---------------------------------
def _hist_or_raise(a):
    if a is None:
        raise RuntimeError("histories are not mirrored on the host (backend history='none')")
    return a


def state(ws, step_or_updt=None):
    if isinstance(ws, CUDAGlobalWorkspace):
        if step_or_updt is None:
            return ws.sub_ws.state
        if hasattr(step_or_updt, "mcmciter"):
            return _hist_or_raise(ws.sub_ws.state_history)[step_or_updt.mcmciter - 1, step_or_updt.pidx - 1]
        return ws.sub_ws.state[np.asarray(step_or_updt.coords) - 1]     # state(ws, updt)
    return ws.sub_ws.state


def state_prop(ws, step=None):                                   # state°
    if isinstance(ws, CUDAGlobalWorkspace):
        return _hist_or_raise(ws.sub_ws.state_proposal_history)[step.mcmciter - 1, step.pidx - 1]
    return ws.sub_ws_prop.state


def num_mcmc_steps(ws):
    return ws.M


def num_updt(ws):
    return ws.NU


def estim_mean(ws):
    return ws.stats()["mean"]


def estim_cov(ws):
    return ws.stats()["cov"]


def ll(ws, i=None):
    return ws.sub_ws.ll if i is None else _hist_or_raise(ws.sub_ws.ll_history)[i - 1]


def ll_prop(ws, i=None):                                         # ll°
    # NB the reference's ll°(ws, i) ignores i and returns the current ll° (workspaces.jl:337);
    # here the i-th proposal log-likelihood is returned.
    return ws.sub_ws_prop.ll if i is None else _hist_or_raise(ws.sub_ws_prop.ll_history)[i - 1]


def accepted(ws, i):
    return _hist_or_raise(ws.acceptance_history)[i - 1]


def set_accepted_(ws, i, v):                                     # set_accepted! workspaces.jl:299-303
    """Overwrite the host mirror of acceptance_history[i] (the device keeps its own record)."""
    _hist_or_raise(ws.acceptance_history)[i - 1] = v


def llr(ws, i):                                                  # workspaces.jl:378
    return np.sum(ll_prop(ws, i) - ll(ws, i), axis=0)


def name_of_update(ws):
    return ws.updt_name


def summary(ws, init=False, file=None):                          # workspaces.jl:244-262
    import sys
    out = file or sys.stdout
    print("Number of MCMC iterations: ", num_mcmc_steps(ws), file=out)
    if init:
        print("Initial θ guess: ", ws.theta_init[:, 0] if ws.C > 0 else [], f"(x {ws.C} chains)", file=out)
        print("Number of updates at each MCMC iteration: ", num_updt(ws), file=out)
        print("Chosen `GlobalWorkspace:` ", type(ws).__name__, file=out)
    else:
        st = ws.stats()
        print("Estimated E[θ] (mean over chains): ", st["mean"].mean(axis=-1), file=out)
        print("Estimated Cov[θ] (mean over chains): ", file=out)
        print(st["cov"].mean(axis=-1), file=out)
