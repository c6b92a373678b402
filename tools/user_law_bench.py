"""User-defined device laws against the built-in sweep, at the shape of BASELINE cfg 2 (4096 chains,
1e6 observations, the two adaptive uniform walks of bench.py): the built-in GSN_IID_1D law and its
DeviceLaw restatement (tests/user_laws.py) in one process, alternating, each timed step after the L2
flush bench.py uses.  Reports ms per iteration, chain-step x observation per second, the instrumented
sweep time per launch, the cold and cached JIT compile time, and a Poisson-regression DeviceLaw at
d = 8 (4096 chains, 1e6 rows) in ms per iteration.  The forward arm runs MALA on the same Poisson
regression (two MALA updates of 4 coordinates) with the hand-written gradient (tests/user_laws.py)
and with forward-mode gradients (tests/user_laws_forward.py), alternating: ms per iteration and
gradient-sweep ms per launch of each.  The chunked arm (--chunked) runs the same MALA problem at
d = 32 and d = 64 (two MALA updates of d/2 coordinates) with the hand-written gradient and with chunked
forward-mode gradients at the library's chunk width, and at d = 8 at chunk widths 8 (unchunked), 4
and 2, each set alternating in one process.  The theta-term arm (--theta-term) runs BASELINE cfg 4
(8192 chains, 8 groups x 4096 rows, MALA on theta_1..8 and two walks, bench.py's updates, 10 iterations per
extmcmc_run_block) on the built-in HIER_NORMAL law with its data-sum cache off and on, and on its
DeviceLaw restatement with a theta term (tests/user_laws_theta.py) with the hand-written and the
forward-mode gradient, alternating: ms per iteration and sweep ms per launch of each.  One JSON object
on stdout (and in --out), with the card's name and power limit read in the same process.

    python tools/user_law_bench.py [--steps 300] [--warmup 30] [--reps 3] [--forward-only]
                                   [--forward-steps 30] [--chunked] [--chunked-steps 6]
                                   [--theta-term] [--theta-steps 50] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (cfg 2 data, updates, initial state, step arrays, timed loop)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make(em, law, x, ups, th0, **bk):
    from extensiblemcmc_jl_b200.mcmc import init_
    mcmc = em.MCMC(ups, backend=em.CUDAMCMCBackend(n_chains=th0.shape[1], seed=3, history="none", **bk))
    init_(mcmc, 1, dict(P=law, obs=x), th0)
    return mcmc.workspace


def sweep_ms(ws, _abi, K):
    lib, h = ws.lib, ws.handle
    msw, nl = ctypes.c_float(), ctypes.c_int64()
    ws._ck(lib.extmcmc_run_block(h, bench.steps_for(None, _abi, 1, 5), 5 * bench.NU))
    ws.sync()
    ws._ck(lib.extmcmc_get_sweep_time(h, ctypes.byref(msw), ctypes.byref(nl)))
    it = 6
    for _ in range(K):
        ws._ck(lib.extmcmc_flush_l2(h))
        ws._ck(lib.extmcmc_run_block(h, bench.steps_for(None, _abi, it, 1), bench.NU))
        it += 1
    ws.sync()
    ws._ck(lib.extmcmc_get_sweep_time(h, ctypes.byref(msw), ctypes.byref(nl)))
    return msw.value / max(nl.value, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--forward-steps", type=int, default=30, help="timed steps of each forward-arm rep")
    ap.add_argument("--forward-only", action="store_true", help="only the forward arm")
    ap.add_argument("--chunked", action="store_true", help="only the chunked arm")
    ap.add_argument("--chunked-steps", type=int, default=6, help="timed steps of each chunked-arm rep")
    ap.add_argument("--theta-term", action="store_true", help="only the theta-term arm (cfg 4)")
    ap.add_argument("--theta-steps", type=int, default=50, help="timed iterations of each theta-term rep")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import extensiblemcmc_jl_b200 as em
    from extensiblemcmc_jl_b200 import _abi
    from tests import user_laws as ul

    out = {"card": card()}
    if args.theta_term:
        theta_term_arm(args, em, _abi, out)
    elif args.chunked:
        chunked_arm(args, em, _abi, out)
    else:
        if not args.forward_only:
            builtin_arms(args, em, _abi, ul, out)
        forward_arm(args, em, _abi, out)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def poisson_problem(em, N, C, d=8):
    """Poisson regression with log link, intercept + d - 1 covariates: rows, initial state."""
    rng = np.random.default_rng(5)
    X = np.empty((N, d))
    X[:, :d - 1] = rng.standard_normal((N, d - 1)) / np.sqrt(d - 1)
    beta = 0.3 * rng.standard_normal(d)
    X[:, d - 1] = rng.poisson(np.exp(beta[0] + X[:, :d - 1] @ beta[1:]))
    thp = beta[:, None] + 1e-3 * rng.standard_normal((d, C))
    return X, thp


def mala_arms(args, em, _abi, d, laws, steps):
    """Poisson regression at d under two MALA updates of d/2 coordinates, 4096 chains x 1e6 rows: every
    law of `laws` (name -> DeviceLaw) in one process, alternating; ms per iteration and per gradient sweep."""
    C, N = bench.CHAINS_PER_GPU, 1_000_000
    X, thp = poisson_problem(em, N, C, d)
    h = d // 2
    ups = lambda: [em.MALAUpdate(1e-3, list(range(1, h + 1))), em.MALAUpdate(1e-3, list(range(h + 1, d + 1)))]  # noqa: E731
    res = {"workload": f"Poisson regression d = {d}, 4096 chains x 1e6 rows, 2 MALA updates of {h} coordinates "
                       "(one gradient sweep each per iteration)"}
    ws = {k: make(em, law, X, ups(), thp, block_len=bench.NU) for k, law in laws.items()}
    times = {k: [] for k in ws}
    for _ in range(args.reps):                           # alternating, the same warm-up each time
        for k, w in ws.items():
            times[k].append(bench.timed_steps(w, _abi, C, steps, 3) / steps)
    for k, w in ws.items():
        res[k] = {"ms_per_iter": float(np.median(times[k])), "ms_per_iter_reps": times[k],
                  "variant": w.lib.extmcmc_sweep_variant_name(w.handle).decode(),
                  "chunk": getattr(laws[k], "chunk", None)}
        w.close()
    for k, law in laws.items():
        wi = make(em, law, X, ups(), thp, block_len=5 * bench.NU, use_graphs=False, instrument=True)
        res[k]["grad_sweep_ms"] = sweep_ms(wi, _abi, max(steps // 3, 3))
        wi.close()
    return res


def chunked_arm(args, em, _abi, out):
    from tests import user_laws as ul
    from tests import user_laws_forward as uf
    for d in (32, 64):
        laws = {"hand": em.DeviceLaw(ul.POISSON_REG, d, d, gradient=True),
                "chunked": em.DeviceLaw(uf.POISSON_REG, d, d, gradient="forward", chunk="auto")}
        res = mala_arms(args, em, _abi, d, laws, args.chunked_steps)
        res["chunked_over_hand_iter"] = res["chunked"]["ms_per_iter"] / res["hand"]["ms_per_iter"]
        res["chunked_over_hand_sweep"] = res["chunked"]["grad_sweep_ms"] / res["hand"]["grad_sweep_ms"]
        out[f"poisson_reg_d{d}_mala"] = res
    d = 8
    laws = {"hand": em.DeviceLaw(ul.POISSON_REG, d, d, gradient=True)}
    laws.update({f"forward_k{k}": em.DeviceLaw(uf.POISSON_REG, d, d, gradient="forward", chunk=k) for k in (8, 4, 2)})
    out["poisson_reg_d8_mala_widths"] = mala_arms(args, em, _abi, d, laws, args.forward_steps)


def forward_arm(args, em, _abi, out):
    from tests import user_laws as ul
    from tests import user_laws_forward as uf
    d = 8
    laws = {"hand": em.DeviceLaw(ul.POISSON_REG, d, d, gradient=True),
            "forward": em.DeviceLaw(uf.POISSON_REG, d, d, gradient="forward")}
    res = mala_arms(args, em, _abi, d, laws, args.forward_steps)
    res["forward_over_hand_iter"] = res["forward"]["ms_per_iter"] / res["hand"]["ms_per_iter"]
    res["forward_over_hand_sweep"] = res["forward"]["grad_sweep_ms"] / res["hand"]["grad_sweep_ms"]
    out["poisson_reg_d8_mala"] = res


def theta_term_arm(args, em, _abi, out):
    """BASELINE cfg 4 on the built-in HIER_NORMAL law (data-sum cache off / on) and on its DeviceLaw
    restatement with a theta term (hand-written / forward-mode gradient), alternating."""
    from extensiblemcmc_jl_b200.mcmc import init_
    from tests import user_laws_theta as ut
    C, G, ng, ipb = 8192, 8, 4096, bench.CFG4_BLOCK_ITERS
    rng = np.random.default_rng(5)                       # bench.py's cfg 4 data, updates and initial state
    tg = rng.standard_normal(G)
    yv = np.concatenate([tg[g] + rng.standard_normal(ng) for g in range(G)])
    grp = np.repeat(np.arange(G), ng)
    rows = np.stack([yv, grp.astype(np.float64)], axis=1)
    ups = lambda: [  # noqa: E731
        em.MALAUpdate(0.02, list(range(1, G + 1)), adpt=em.AdaptationMALA(adapt_every_k_steps=50, scale=1e-3, min=1e-5)),
        em.RandomWalkUpdate(em.UniformRandomWalk([0.3]), [G + 1], adpt=em.AdaptationUnifRW([0.0], adapt_every_k_steps=50, scale=0.02)),
        em.RandomWalkUpdate(em.UniformRandomWalk([0.3], [True]), [G + 2], prior=em.ImproperPosPrior(),
                            adpt=em.AdaptationUnifRW([0.0], adapt_every_k_steps=50, scale=0.02))]
    th0 = np.concatenate([np.zeros(G), [0.0, 1.0]])
    P = G + 2
    arms = {"builtin_no_cache": (dict(P=em.HierNormalLaw(G), obs=yv, groups=grp), "0"),
            "builtin_cache": (dict(P=em.HierNormalLaw(G), obs=yv, groups=grp), "1"),
            "device_law_hand": (dict(P=em.DeviceLaw(ut.HIER_HAND, P, 2, gradient=True, theta_term=True), obs=rows), None),
            "device_law_forward": (dict(P=em.DeviceLaw(ut.HIER_FORWARD, P, 2, gradient="forward", theta_term=True),
                                        obs=rows), None)}
    out["theta_term_workload"] = (f"BASELINE cfg 4: hierarchical normal, {G} groups x {ng} rows, {C} chains, MALA(theta_1..8) "
                                  f"+ RW(mu) + RW-pos(tau), {ipb} iterations per extmcmc_run_block")
    warm = 3 * ipb
    steps = -(-args.theta_steps // ipb) * ipb

    def make(data, cache, **bk):
        # EXTMCMC_DATA_CACHE is read when the sweep is planned: on the first block of the handle
        os.environ["EXTMCMC_DATA_CACHE"] = cache or "1"
        mcmc = em.MCMC(ups(), backend=em.CUDAMCMCBackend(n_chains=C, seed=7, history="none", block_len=3 * ipb, **bk))
        init_(mcmc, 1, data, th0)
        w = mcmc.workspace
        bench._generic_timed(w, _abi, 3, 0, warm, ipb=ipb)
        return w
    ws = {k: make(d, cache) for k, (d, cache) in arms.items()}
    it = {k: warm + 1 for k in ws}
    times = {k: [] for k in ws}
    for _ in range(args.reps):                           # alternating
        for k, w in ws.items():
            times[k].append(bench._generic_timed(w, _abi, 3, steps, 0, it0=it[k], ipb=ipb) / steps)
            it[k] += steps
    res = {}
    for k, w in ws.items():
        res[k] = {"ms_per_iter": float(np.median(times[k])), "ms_per_iter_reps": times[k],
                  "variant": w.lib.extmcmc_sweep_variant_name(w.handle).decode()}
        w.close()
    for k, (d, cache) in arms.items():
        wi = make(d, cache, use_graphs=False, instrument=True)
        msw, nl = ctypes.c_float(), ctypes.c_int64()
        wi._ck(wi.lib.extmcmc_get_sweep_time(wi.handle, ctypes.byref(msw), ctypes.byref(nl)))
        bench._generic_timed(wi, _abi, 3, 2 * ipb, 0, it0=warm + 1, ipb=ipb)
        wi._ck(wi.lib.extmcmc_get_sweep_time(wi.handle, ctypes.byref(msw), ctypes.byref(nl)))
        res[k]["sweep_ms_per_launch"] = msw.value / max(nl.value, 1)
        res[k]["sweep_launches_per_iter"] = nl.value / (2 * ipb)
        wi.close()
    os.environ.pop("EXTMCMC_DATA_CACHE", None)
    for k in ("device_law_hand", "device_law_forward"):
        res[k + "_over_builtin_cache"] = res[k]["ms_per_iter"] / res["builtin_cache"]["ms_per_iter"]
        res[k + "_over_builtin_no_cache"] = res[k]["ms_per_iter"] / res["builtin_no_cache"]["ms_per_iter"]
    out["hier_cfg4_theta_term"] = res


def builtin_arms(args, em, _abi, ul, out):
    out["workload"] = "BASELINE cfg 2 shape: 4096 chains x 1e6 observations, 2 adaptive uniform walks"
    t0 = time.perf_counter()
    user_gsn = em.DeviceLaw(ul.GSN1D, 2, 1)              # cold: NVRTC + ptxas of every instantiation
    out["jit_cold_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    em.DeviceLaw(ul.GSN1D, 2, 1)                         # the same input again: the process-wide cache
    out["jit_cached_s"] = time.perf_counter() - t0

    x = bench.cfg2_data()
    C, N, NU = bench.CHAINS_PER_GPU, x.shape[0], bench.NU
    th0 = bench.cfg2_theta_init(x, C)
    ws = {"builtin": make(em, em.GsnTargetLaw([0.0]), x, bench.cfg2_updates(em), th0, block_len=NU),
          "device_law": make(em, user_gsn, x[:, None], bench.cfg2_updates(em), th0, block_len=NU)}
    out["variant"] = {k: w.lib.extmcmc_sweep_variant_name(w.handle).decode() for k, w in ws.items()}
    times = {k: [] for k in ws}
    for _ in range(args.reps):                           # alternating, the same warm-up each time
        for k, w in ws.items():
            times[k].append(bench.timed_steps(w, _abi, C, args.steps, args.warmup) / args.steps)
    for k, w in ws.items():
        ms = float(np.median(times[k]))
        out[k] = {"ms_per_iter": ms, "ms_per_iter_reps": times[k],
                  "chain_step_obs_per_s": C * NU * N / (ms * 1e-3)}
        w.close()
    for k, law, xx in (("builtin", em.GsnTargetLaw([0.0]), x), ("device_law", user_gsn, x[:, None])):
        wi = make(em, law, xx, bench.cfg2_updates(em), th0, block_len=5 * NU, use_graphs=False, instrument=True)
        out[k]["sweep_ms"] = sweep_ms(wi, _abi, args.steps // 3)
        wi.close()
    out["device_over_builtin"] = out["device_law"]["ms_per_iter"] / out["builtin"]["ms_per_iter"]

    # Poisson regression with log link, d = 8 (intercept + 7 covariates), two uniform walks of 4 coordinates
    d = 8
    X, thp = poisson_problem(em, N, C, d)
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([1e-3] * 4), [1, 2, 3, 4]),
           em.RandomWalkUpdate(em.UniformRandomWalk([1e-3] * 4), [5, 6, 7, 8])]
    t0 = time.perf_counter()
    preg = em.DeviceLaw(ul.POISSON_REG, d, d)
    jit = time.perf_counter() - t0
    wp = make(em, preg, X, ups, thp, block_len=NU)
    tp = [bench.timed_steps(wp, _abi, C, args.steps, args.warmup) / args.steps for _ in range(args.reps)]
    out["poisson_reg_d8"] = {"ms_per_iter": float(np.median(tp)), "ms_per_iter_reps": tp, "jit_cold_s": jit,
                             "variant": wp.lib.extmcmc_sweep_variant_name(wp.handle).decode(),
                             "chain_step_obs_per_s": C * NU * N / (float(np.median(tp)) * 1e-3)}
    wp.close()


if __name__ == "__main__":
    main()
