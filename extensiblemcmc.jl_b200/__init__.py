"""extmcmc-cuda: B200-native transition-step engine behind ExtensibleMCMC.jl's backend API.

Python host mirror of the reference's user-facing API (src/ExtensibleMCMC.jl:31-41 exports)
for the hot path only.  Julia names map as: `f!` -> `f_`, `x°` -> `x_prop`.
"""
from .types import (MCMCUpdate, MCMCParamUpdate, MCMCGradientBasedUpdate, MCMCBackend,
                    GenericMCMCBackend, GlobalWorkspace, LocalWorkspace, PRESTEP, POSTSTEP,
                    PreMCMCStep, PostMCMCStep)
from .schedule import MCMCSchedule, Step, reschedule_
from .random_walk import UniformRandomWalk, GaussianRandomWalk, GaussianRandomWalkMix
from .adaptation import (NoAdaptation, AdaptationUnifRW, HaarioTypeAdaptation, AdaptationMALA,
                         isequal_except)
from .priors import (Prior, ImproperPrior, ImproperPosPrior, StandardPrior, ProductPrior,
                     Normal, Gamma, Uniform, Exponential, InverseGamma, Beta, LogNormal, Cauchy, MvNormal,
                     DevicePrior)
from .updates import RandomWalkUpdate, MALAUpdate, HamiltonianMCUpdate
from .gsn_target import GsnTargetLaw
from .hier_normal import HierNormalLaw
from .logistic import LogisticLaw
from .device_law import DeviceLaw
from .workspaces import (CUDAMCMCBackend, CUDAGlobalWorkspace, CUDALocalWorkspace,
                         DeviceGeneratedObs, init_global_workspace, create_workspace,
                         create_workspaces, state, state_prop, ll, ll_prop, accepted, set_accepted_, llr,
                         estim_mean, estim_cov, num_mcmc_steps, num_updt, name_of_update, summary)
from .callbacks import Callback, SavingCallback, REPLCallback
from .mcmc import MCMC, init_
from .run import run_
from .ess import ess_geyer
