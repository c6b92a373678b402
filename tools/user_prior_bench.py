"""User-defined priors (DevicePrior) against the built-in priors, arms alternating in one process.

Logistic arm: BASELINE cfg 3 as bench.py runs it (LogisticLaw, d = 256 features, 1024 chains x 1e6 rows,
MALA with bench.py's step and adaptation, the logistic FP64-DMMA sweep).  A user prior covers at most 64
coordinates, so every arm runs the 256 coordinates as four MALA updates of 64 (four sweeps per iteration
against cfg 3's one): StandardPrior(Normal(0, 10)), its DevicePrior restatement (tests/user_priors.py,
hand-written gradient) and a Laplace(0, 1) DevicePrior: ms per iteration (four updates) of each.  MALA runs
the prior's gradient kernel on the current state and on the proposal; the likelihood sweep is unchanged.

Forward-mode arm: LogisticLaw d = 16 with few rows (--fwd-n-obs), one MALA update of all 16 coordinates:
StandardPrior(Normal(0, 10)), its restatement with logprior_grad and in forward mode (the 16 Dual<16>
arguments of the forward kernel live in local memory, 2176 bytes per thread): ms per iteration.

Step-kernel arm: GsnTargetLaw d = 1 with few observations (--small-n-obs), so that the step kernels, not
the sweep, take the time: one uniform walk on (mu, sigma^2) with StandardPrior(Normal) and with its
restatement: ms per update step.  A user prior adds its kernel per element and its proposal no longer
rides on the previous accept kernel.

One JSON object on stdout (and in --out), with the card's name and power limit read in the same process.

    python tools/user_prior_bench.py [--reps 3] [--logi-iters 20] [--small-iters 2000] [--out FILE]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import extensiblemcmc_jl_b200 as em  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from tests import user_priors as up  # noqa: E402
from tests.parity import GpuSession  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def session(law, ups, obs, th0, Cn, y=None, block=100):
    g = GpuSession(law, ups, obs, th0, Cn, y=y, n_steps_hint=block, use_graphs=1)
    for i, u in enumerate(ups):
        if hasattr(u.prior, "abi_attach"):
            g.ck(u.prior.abi_attach(g.lib, g.h, i))
    return g


def timed(g, steps, block):
    """ms per schedule element over `steps`, run in blocks of `block` elements, ending in a device sync"""
    arrs = [orc.steps_array(steps[b:b + block]) for b in range(0, len(steps), block)]
    g.ck(g.lib.extmcmc_sync(g.h))
    t0 = time.perf_counter()
    for a in arrs:
        g.ck(g.lib.extmcmc_run_block(g.h, a, len(a)))
    g.ck(g.lib.extmcmc_sync(g.h))
    return (time.perf_counter() - t0) * 1e3 / len(steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--logi-chains", type=int, default=1024)
    ap.add_argument("--logi-n-obs", type=int, default=1_000_000)
    ap.add_argument("--logi-iters", type=int, default=20)
    ap.add_argument("--fwd-chains", type=int, default=4096)
    ap.add_argument("--fwd-n-obs", type=int, default=1024)
    ap.add_argument("--fwd-iters", type=int, default=500)
    ap.add_argument("--small-chains", type=int, default=4096)
    ap.add_argument("--small-n-obs", type=int, default=256)
    ap.add_argument("--small-iters", type=int, default=2000)
    ap.add_argument("--out")
    a = ap.parse_args()
    out = dict(card=card())

    d = 256
    rng = np.random.default_rng(4)
    X = rng.standard_normal((a.logi_n_obs, d)) / math.sqrt(d)
    beta = rng.standard_normal(d)
    y = (rng.random(a.logi_n_obs) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
    th0 = 0.01 * np.random.default_rng(40).standard_normal((d, a.logi_chains))
    arms = {
        "builtin_normal": em.StandardPrior(em.Normal(0.0, 10.0)),
        "device_normal": em.DevicePrior(up.NORMAL, gradient=True, params=(0.0, 10.0)),
        "device_laplace": em.DevicePrior(up.LAPLACE, gradient=True, params=(0.0, 1.0)),
    }
    NU = 4
    steps = list(em.MCMCSchedule(a.logi_iters + 2, NU))
    mala = lambda p, q: em.MALAUpdate(0.02, list(range(64 * q + 1, 64 * q + 65)), prior=p,
                                      adpt=em.AdaptationMALA(adapt_every_k_steps=20, scale=1e-3, min=1e-5, offset=2.0))
    sess = {k: session(em.LogisticLaw(d), [mala(p, q) for q in range(NU)], X, th0, a.logi_chains, y=y,
                       block=len(steps)) for k, p in arms.items()}
    for g in sess.values():
        timed(g, steps[:2 * NU], 2 * NU)             # warm-up: graph capture, module load
    res = {k: [] for k in arms}
    for _ in range(a.reps):
        for k, g in sess.items():
            res[k].append(NU * timed(g, steps[2 * NU:], len(steps) - 2 * NU))
    out["logistic_d256_4x64_mala_ms_per_iter"] = {k: dict(median=float(np.median(v)), all=v) for k, v in res.items()}
    out["logistic_shape"] = dict(d=d, chains=a.logi_chains, n_obs=a.logi_n_obs, iters=a.logi_iters)
    for g in sess.values():
        g.close()

    d = 16
    X = rng.standard_normal((a.fwd_n_obs, d)) / math.sqrt(d)
    beta = rng.standard_normal(d)
    y = (rng.random(a.fwd_n_obs) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
    th0 = 0.01 * np.random.default_rng(41).standard_normal((d, a.fwd_chains))
    arms = {
        "builtin_normal": em.StandardPrior(em.Normal(0.0, 10.0)),
        "device_normal_hand": em.DevicePrior(up.NORMAL, gradient=True, params=(0.0, 10.0)),
        "device_normal_forward": em.DevicePrior(up.NORMAL_FORWARD, gradient="forward", params=(0.0, 10.0)),
    }
    block = 100
    steps = list(em.MCMCSchedule(a.fwd_iters + block, 1))
    sess = {k: session(em.LogisticLaw(d), [em.MALAUpdate(0.05, list(range(1, d + 1)), prior=p)], X, th0,
                       a.fwd_chains, y=y, block=block) for k, p in arms.items()}
    for g in sess.values():
        timed(g, steps[:block], block)
    res = {k: [] for k in arms}
    for _ in range(a.reps):
        for k, g in sess.items():
            res[k].append(timed(g, steps[block:], block))
    out["logistic_d16_mala_ms_per_iter"] = {k: dict(median=float(np.median(v)), all=v) for k, v in res.items()}
    out["logistic_d16_shape"] = dict(d=d, chains=a.fwd_chains, n_obs=a.fwd_n_obs, iters=a.fwd_iters, block=block)
    for g in sess.values():
        g.close()

    x = 1.0 + rng.standard_normal(a.small_n_obs)
    th0 = np.array([1.0, 1.0])
    arms = {
        "builtin_normal": em.StandardPrior(em.Normal(0.0, 10.0)),
        "device_normal": em.DevicePrior(up.NORMAL, params=(0.0, 10.0), n_coords=2),
    }
    block = 100
    steps = list(em.MCMCSchedule(a.small_iters + block, 1))
    sess = {k: session(em.GsnTargetLaw([0.0]),
                       [em.RandomWalkUpdate(em.UniformRandomWalk([0.1, 0.1], [False, True]), [1, 2], prior=p)],
                       x, th0, a.small_chains, block=block) for k, p in arms.items()}
    for g in sess.values():
        timed(g, steps[:block], block)
    res = {k: [] for k in arms}
    for _ in range(a.reps):
        for k, g in sess.items():
            res[k].append(timed(g, steps[block:], block))
    out["gsn1d_small_ms_per_step"] = {k: dict(median=float(np.median(v)), all=v) for k, v in res.items()}
    out["gsn1d_shape"] = dict(chains=a.small_chains, n_obs=a.small_n_obs, steps=a.small_iters, block=block)
    for g in sess.values():
        g.close()
    s = json.dumps(out)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
