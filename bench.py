#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE cfg 2.

    python bench.py --gpus N --steps K --warmup W            (N > 1: under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --steps K --warmup W --dump-outputs DIR  (also writes DIR/<name>.npy, see dump_outputs)

metric   chain-steps x observations / second.  One chain-step = one (mcmciter, pidx)
         schedule element for one chain = one full-data log-likelihood evaluation
         (reference: src/run.jl:257).
step     one MCMC iteration of cfg 2 = its 2 random-walk updates for all chains, i.e.
         2 * C * N chain-step x observation units.
value    device-resident throughput: K steps timed with CUDA events on the library's own
         stream, L2 flushed (untimed) before every step, max over ranks.
e2e      the whole cfg 2 job through the reference-facing API `run_(mcmc, M, data, theta0)`
         with host buffers: observation upload, every block launch, and the copy of every
         history row back to the host are inside the timed region.
extra    sub-records of the same JSON line: `strong_cfg5` (BASELINE cfg 5: N = 1e9 observations
         sharded over the ranks, NCCL all-reduce and the library's fused NVLink exchange, with an
         in-run cross-rank parity check), `cfg4` (hierarchical model with the mixed MALA /
         random-walk schedule, 8192 chains per GPU, i.e. BASELINE's 65536 chains at N = 8; at
         N = 1 with and without the data-sum cache) and at N = 1 `cfg3` (logistic regression on
         the FP64 tensor path).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line.  NCCL's INFO log (communicator lines with `nranks N`) goes
# to stderr instead of being silenced, so the ranks of every communicator stay observable.
# (the image presets NCCL_DEBUG=VERSION, so this is an override, not a default; EXTMCMC_NCCL_DEBUG picks another level)
os.environ["NCCL_DEBUG"] = os.environ.get("EXTMCMC_NCCL_DEBUG", "INFO")
os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"

N_OBS = 1_000_000
CHAINS_PER_GPU = 4096
NU = 2
# cfg 4 is timed in blocks of this many iterations per extmcmc_run_block (see measure_cfg34)
CFG4_BLOCK_ITERS = 10


def cfg2_data():
    return 1.5 + 2.0 * np.random.default_rng(2).standard_normal(N_OBS)


def cfg2_updates(em):
    mk = lambda: em.AdaptationUnifRW([0.0], adapt_every_k_steps=50, target_accpt_rate=0.234,
                                     scale=5e-4, min=1e-7, max=1e7, offset=100.0)
    return [em.RandomWalkUpdate(em.UniformRandomWalk([5e-3]), [1], adpt=mk()),
            em.RandomWalkUpdate(em.UniformRandomWalk([5e-3], [True]), [2],
                                prior=em.ImproperPosPrior(), adpt=mk())]


def cfg2_theta_init(x, n_chains, offset=0):
    rng = np.random.default_rng(3)
    z = rng.standard_normal((2, offset + n_chains))[:, offset:]
    th = np.empty((2, n_chains))
    th[0] = x.mean() + 0.01 * z[0]
    th[1] = x.var(ddof=1) * np.exp(0.01 * z[1])
    return th


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region: NVML polled every 20 ms
    from a thread of this process (nvidia-smi -lms as the fallback; same counters).  A timed region
    shorter than a few sampling periods is followed by an untimed continuation of the very same
    steps (`extend`) until three samples under load exist; the JSON says so in `window`."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.idx, self.proc, self.rows = gpu_index, None, []     # rows: (sm, sm_max, watts, reasons)
        self.nv, self.dev, self.run, self.t = None, None, False, None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.idx).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.idx)

    def start(self):
        self.run = True
        try:
            self.nv, self.dev = self._nvml_handle()
            self._sample_nvml()                                  # fails here, not in the thread
            self.rows.clear()
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read_smi, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _sample_nvml(self):
        nv, d = self.nv, self.dev
        sm = float(nv.nvmlDeviceGetClockInfo(d, nv.NVML_CLOCK_SM))
        smax = float(nv.nvmlDeviceGetMaxClockInfo(d, nv.NVML_CLOCK_SM))
        watts = nv.nvmlDeviceGetPowerUsage(d) / 1000.0
        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(d)
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        self.rows.append((sm, smax, watts, {k for k, b in bits.items() if mask & b}))

    def _poll_nvml(self):
        while self.run:
            try:
                self._sample_nvml()
            except Exception:
                pass
            time.sleep(0.02)

    def _read_smi(self):
        for line in self.proc.stdout:
            f = [v.strip() for v in line.split(",")]
            if len(f) < 9:
                continue
            try:
                self.rows.append((float(f[1]), float(f[2]), float(f[3]),
                                  {nm for nm, v in zip(self.NAMES, f[5:9]) if v.lower().startswith("active")}))
            except ValueError:
                continue

    def stop(self, extend=None):
        if self.nv is None and not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        n_timed = len(self.rows)
        window = "timed region"
        if extend is not None and n_timed < 3:
            t_end = time.monotonic() + 2.0
            while len(self.rows) < 3 and time.monotonic() < t_end:
                extend()
            window = "timed region + untimed continuation of the same steps (region shorter than 3 samples)"
        self.run = False
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self.t is not None:
            self.t.join(timeout=1.0)
        rows = list(self.rows)
        reasons = set().union(*[r[3] for r in rows]) if rows else set()
        return {"sm_mhz": float(np.median([r[0] for r in rows])) if rows else None,
                "sm_max_mhz": float(max(r[1] for r in rows)) if rows else None,
                "power_w_max": float(max(r[2] for r in rows)) if rows else None,
                "samples": len(rows), "samples_in_timed_region": n_timed, "window": window,
                "source": "nvml" if self.nv is not None else "nvidia-smi", "reasons": sorted(reasons)}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


def steps_for(em, _abi, it0, n_iters):
    """ABI step array for iterations it0 .. it0 + n_iters - 1 of the 2-update schedule."""
    arr = (_abi.Step * (n_iters * NU))()
    k = 0
    for it in range(it0, it0 + n_iters):
        for pj in range(NU):
            arr[k].mcmciter = it
            arr[k].pidx = pj
            first = (it == 1 and pj == 0)
            arr[k].prev_pidx = -1 if first else (pj - 1 if pj else NU - 1)
            arr[k].prev_mcmciter = 0 if first else (it if pj else it - 1)
            k += 1
    return arr


def make_ws(em, x, n_chains, chain_offset, device, **bk):
    from extensiblemcmc_jl_b200.mcmc import init_
    ups = cfg2_updates(em)
    mcmc = em.MCMC(ups, backend=em.CUDAMCMCBackend(n_chains=n_chains, device=device, seed=3,
                                                   chain_offset=chain_offset, history="none", **bk))
    init_(mcmc, 1, dict(P=em.GsnTargetLaw([0.0]), obs=x), cfg2_theta_init(x, n_chains, chain_offset))
    return mcmc.workspace


def timed_steps(ws, _abi, C, K, W, flush=True, it0=1):
    """W warm-up + K timed steps (one MCMC iteration each, iterations it0, it0 + 1, ...).  Every
    timed step is bracketed by its own CUDA event pair on the library stream (the L2 flush before
    it is outside the pair); nothing synchronises the host inside the loop.  Returns the summed
    device ms."""
    import ctypes
    lib, h = ws.lib, ws.handle
    it = it0
    for _ in range(W):
        ws._ck(lib.extmcmc_run_block(h, steps_for(None, _abi, it, 1), NU)); it += 1
    ws.sync()
    total = 0.0
    ms = ctypes.c_float()
    done = 0
    while done < K:
        n = min(K - done, 2048)
        for k in range(n):
            if flush:
                ws._ck(lib.extmcmc_flush_l2(h))
            ws._ck(lib.extmcmc_event_record(h, 2 * k))
            ws._ck(lib.extmcmc_run_block(h, steps_for(None, _abi, it, 1), NU))
            ws._ck(lib.extmcmc_event_record(h, 2 * k + 1))
            it += 1
        ws.sync()
        for k in range(n):
            ws._ck(lib.extmcmc_event_elapsed(h, 2 * k, 2 * k + 1, ctypes.byref(ms)))
            total += ms.value
        done += n
    return total


def last_step_outputs(ws, _abi, n_iters):
    """What a caller of the timed path receives after its last step (iteration n_iters, both
    updates), as float64 arrays with the chain axis last: the chain state and its log-likelihood,
    that iteration's proposals, their log-likelihoods and the accept decisions (from the device
    history ring), the step size of every update and the running chain statistics."""
    p, C = ws.p, ws.C
    theta, ll = ws.refresh_state()
    prop, llp, acc = np.empty((NU, p, C)), np.empty((NU, C)), np.empty((NU, C), dtype=np.uint8)
    ws._ck(ws.lib.extmcmc_get_history(ws.handle, (n_iters - 1) * NU, n_iters * NU, None, _abi.dptr(prop), None,
                                      _abi.dptr(llp), acc.ctypes.data_as(_abi.c_uint8_p)))
    st = ws.stats()
    out = {"theta": theta, "loglik": ll, "theta_prop": prop, "loglik_prop": llp, "accepted": acc,
           "eps": np.concatenate([ws.eps(u) for u in range(1, NU + 1)]),
           "mean": st["mean"], "cov": st["cov"], "rolling_accept_rate": st["rolling_ar"],
           "n_accept": st["n_accept"], "n_prop": st["n_prop"]}
    return {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in out.items()}


def dump_outputs(dirname, arrays, dist=None):
    """Writes dirname/<name>.npy for every array; with several ranks the chains of all ranks are
    gathered (rank order along the chain axis) and rank 0 writes them."""
    if dist is not None:
        import torch
        for k, a in arrays.items():
            t = torch.from_numpy(a).cuda()
            parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
            dist.all_gather(parts, t)
            arrays[k] = torch.cat(parts, dim=-1).cpu().numpy()
        if dist.get_rank() != 0:
            return
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), a)


def ncu_traffic(kernel_substr, csv_name):
    """dram__bytes_read.sum + dram__bytes_write.sum of one kernel launch, read at run time from the
    committed summary of an `ncu --set full` capture (tools/ncu_summary.py) under profiles/."""
    path = os.path.join(ROOT, "profiles", csv_name)
    try:
        import csv
        tot, unit_scale = 0.0, {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        seen = set()
        for row in csv.DictReader(open(path)):
            if kernel_substr in row["kernel"] and row["metric"] in ("dram__bytes_read.sum", "dram__bytes_write.sum") \
                    and row["metric"] not in seen:
                seen.add(row["metric"])
                tot += float(row["value"].replace(",", "")) * unit_scale.get(row["unit"], 1.0)
        if len(seen) == 2:
            return tot, f"profiles/{csv_name} (ncu --set full capture of this kernel at this shape, parsed at run time)"
    except Exception:
        pass
    return None, f"profiles/{csv_name} not found or without dram__bytes rows"


def fp64_peaks(ws, clocks, n_sms=148):
    """FP64 peak two ways: the FMA micro-benchmark run in this process, and lanes x clock
    (SMs x 64 FP64 lanes x 2 flop x the SM clock sampled under load)."""
    import ctypes
    pk = ctypes.c_double()
    ws._ck(ws.lib.extmcmc_measure_fp64_peak(ws.handle, ctypes.byref(pk)))
    mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
    return pk.value, n_sms * 64 * 2 * mhz * 1e6 / 1e12


def measure_cfg5(args, em, _abi, par, dist, rank, world, local, peaks, peak_src):
    """BASELINE cfg 5: ONE dataset of N = 1e9 Gaussian observations generated on the device,
    sharded by observations over the ranks (strong scaling), C = 8 replicated chains, two adaptive
    random-walk updates per iteration.  Per update step the per-chain partial sums of all ranks are
    combined: `nccl` = ncclAllReduce between the sweep and the accept kernel; `p2p` = the library's
    own exchange (stores into every peer over NVLink + flags, inside the persistent block kernel).
    In-run checks: every rank ends in the same state with the same decision counts, and the
    sharded log-likelihood of a 2^24-observation prefix equals the single-rank one."""
    import ctypes
    import torch
    from extensiblemcmc_jl_b200.mcmc import init_
    n_total, C, iters, blk_iters = args.cfg5_n_obs, 8, args.cfg5_iters, 10
    first, cnt = par.shard_obs(n_total, rank, world)
    mk = lambda: em.AdaptationUnifRW([0.0], adapt_every_k_steps=50, target_accpt_rate=0.234,
                                     scale=5e-4 / 30, min=1e-7 / 30, max=1e7, offset=100.0)
    ups = lambda: [em.RandomWalkUpdate(em.UniformRandomWalk([5e-3 / 30]), [1], adpt=mk()),
                   em.RandomWalkUpdate(em.UniformRandomWalk([5e-3 / 30], [True]), [2], prior=em.ImproperPosPrior(), adpt=mk())]
    th0 = np.repeat(np.array([[1.5], [4.0]]), C, axis=1) * (1.0 + 1e-4 * np.arange(C))[None, :]

    def backend(mode, n_chains=C, **kw):
        if world == 1:
            return em.CUDAMCMCBackend(n_chains=n_chains, device=local, seed=6, history="none", **kw)
        extra = {"p2p_allgather": par.p2p_allgather_fn(dist)} if mode == "p2p" else {}
        return par.backend_for_rank(rank, world, local, n_chains, shard="obs", comm_id=par.exchange_comm_id(dist),
                                    seed=6, history="none", **extra, **kw)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    out = {"n_obs_total": n_total, "n_obs_per_gpu": cnt, "chains": C, "iters": iters,
           "block": f"{blk_iters} iterations ({blk_iters * NU} schedule elements) per extmcmc_run_block", "modes": {}}
    for mode in (["single"] if world == 1 else ["nccl", "p2p"]):
        mcmc = em.MCMC(ups(), backend=backend(mode, block_len=blk_iters * NU, use_graphs=True))
        init_(mcmc, 1, dict(P=em.GsnTargetLaw([0.0]), obs=em.DeviceGeneratedObs(cnt, 1.5, 2.0, 6, first)), th0)
        ws = mcmc.workspace
        lib, h = ws.lib, ws.handle
        it = 1
        for _ in range(2):                                     # warm-up: graph capture / first launches
            ws._ck(lib.extmcmc_run_block(h, steps_for(None, _abi, it, blk_iters), blk_iters * NU)); it += blk_iters
        ws.sync()
        sampler = ClockSampler(local)
        barrier()
        sampler.start()
        l0 = lib.extmcmc_launch_count(h)
        ws._ck(lib.extmcmc_event_record(h, 0))
        for _ in range(iters // blk_iters):
            ws._ck(lib.extmcmc_run_block(h, steps_for(None, _abi, it, blk_iters), blk_iters * NU)); it += blk_iters
        ws._ck(lib.extmcmc_event_record(h, 1))
        ws.sync()
        ms = ctypes.c_float()
        ws._ck(lib.extmcmc_event_elapsed(h, 0, 1, ctypes.byref(ms)))
        launches = int(lib.extmcmc_launch_count(h) - l0)
        clocks = sampler.stop()
        t = torch.tensor([ms.value], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        n_it = (iters // blk_iters) * blk_iters
        # every rank must hold the same chains: state and decision counts, bit for bit
        th, ll = ws.refresh_state()
        st = ws.stats()
        sig = np.concatenate([th.ravel(), ll, st["n_accept"].ravel().astype(np.float64)])
        same = True
        if dist is not None:
            g = [torch.zeros(sig.size, dtype=torch.float64, device="cuda") for _ in range(world)]
            dist.all_gather(g, torch.tensor(sig, device="cuda"))
            same = all(bool(torch.equal(g[0], q)) for q in g[1:])
        variant = lib.extmcmc_sweep_variant_name(h).decode()
        ws.close()
        step_s = ms_total * 1e-3 / (n_it * NU)
        gbs = 8.0 * cnt / step_s / 1e9
        out["modes"][mode] = {
            "ms_per_iteration": ms_total / n_it, "value": C * n_it * NU * float(n_total) / (ms_total * 1e-3),
            "unit": "chain-step*obs/s", "kernel": variant, "gpu_launches": launches,
            "hbm_gbs_per_gpu": gbs, "hbm_frac_per_gpu": gbs / peaks["hbm_gbs"], "hbm_peak": peaks["hbm_gbs"],
            "hbm_peak_source": peak_src,
            "hbm_note": "8 B x observations of this rank / whole update-step time (sweep + exchange + decision)",
            "decisions_equal_across_ranks": bool(same), "accept_rate": float(st["n_accept"].sum() / max(st["n_prop"].sum(), 1)),
            "clocks": clocks}
        barrier()
    # ---- sharded vs single-rank log-likelihood on a 2^24-observation prefix --------------------
    n_pre = min(1 << 24, n_total)
    thp = np.repeat(np.array([[1.5], [4.0]]), C, axis=1) * (1.0 + 0.01 * np.arange(C))[None, :]
    if world > 1:
        pf, pc = par.shard_obs(n_pre, rank, world)
        m1 = em.MCMC(ups(), backend=backend("nccl", use_graphs=False))
        init_(m1, 1, dict(P=em.GsnTargetLaw([0.0]), obs=em.DeviceGeneratedObs(pc, 1.5, 2.0, 6, pf)), thp)
        ll_sh = m1.workspace.eval_loglik()
        m1.workspace.close()
        rel = None
        if rank == 0:
            m2 = em.MCMC(ups(), backend=em.CUDAMCMCBackend(n_chains=C, device=local, seed=6, history="none", use_graphs=False))
            init_(m2, 1, dict(P=em.GsnTargetLaw([0.0]), obs=em.DeviceGeneratedObs(n_pre, 1.5, 2.0, 6, 0)), thp)
            ll_1 = m2.workspace.eval_loglik()
            m2.workspace.close()
            rel = float(np.max(np.abs(ll_sh - ll_1) / np.abs(ll_1)))
        out["ll_rel_vs_single_rank"] = rel
        out["ll_check"] = f"extmcmc_eval_loglik on the first 2^24 observations: sharded over {world} ranks (NCCL) vs rank 0 alone"
        barrier()
    return out


def measure_cfg34(args, workload, em, _abi, local, steps, chain_offset=0):
    """BASELINE cfg 3 (logistic regression d = 256, N = 1e6, 1024 chains, MALA, FP64 tensor-core GEMMs)
    or cfg 4 (hierarchical normal, 8 groups x 4096 observations, MALA + 2 random-walk updates, 8192
    chains per GPU) on one GPU: ms per iteration and the roofline of its dominant kernel."""
    import ctypes
    from extensiblemcmc_jl_b200.mcmc import init_
    rng = np.random.default_rng(4 if workload == "cfg3" else 5)
    if workload == "cfg3":
        C, d, N = 1024, 256, args.cfg3_n_obs
        X = rng.standard_normal((N, d)) / np.sqrt(d)
        beta = rng.standard_normal(d)
        y = (rng.random(N) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
        data = dict(P=em.LogisticLaw(d), obs=X, y=y)
        ups = [em.MALAUpdate(0.02, list(range(1, d + 1)), prior=em.StandardPrior(em.Normal(0.0, 10.0)),
                             adpt=em.AdaptationMALA(adapt_every_k_steps=20, scale=1e-3, min=1e-5, offset=2.0))]
        th0 = 0.01 * np.random.default_rng(40).standard_normal((d, C))
        n_obs, flops_per_iter, sweeps_per_iter = N, 4.0 * d * C * N, 1
        desc = f"BASELINE cfg3: logistic regression d={d}, N={N:.3g}, {C} chains/GPU, MALAUpdate on all coordinates"
    else:
        C, G, ng = 8192, 8, 4096
        tg = rng.standard_normal(G)
        yv = np.concatenate([tg[g] + rng.standard_normal(ng) for g in range(G)])
        data = dict(P=em.HierNormalLaw(G), obs=yv, groups=np.repeat(np.arange(G), ng))
        ups = [em.MALAUpdate(0.02, list(range(1, G + 1)), adpt=em.AdaptationMALA(adapt_every_k_steps=50, scale=1e-3, min=1e-5)),
               em.RandomWalkUpdate(em.UniformRandomWalk([0.3]), [G + 1], adpt=em.AdaptationUnifRW([0.0], adapt_every_k_steps=50, scale=0.02)),
               em.RandomWalkUpdate(em.UniformRandomWalk([0.3], [True]), [G + 2], prior=em.ImproperPosPrior(),
                                   adpt=em.AdaptationUnifRW([0.0], adapt_every_k_steps=50, scale=0.02))]
        th0 = np.concatenate([np.zeros(G), [0.0, 1.0]])
        # per iteration: 2 gradient sweeps (3 FP64 instructions per chain x observation: x - mu, the
        # square and the first-order sum) + 2 plain sweeps (2 instructions) = 10 issue slots = 20 "flop"
        # at the FMA rate the peak is quoted in
        # With the data-sum cache (default; EXTMCMC_DATA_CACHE=0 turns it off) the mu / tau elements and
        # the current-state gradient reuse the per-group sums: ONE gradient sweep per iteration (3 slots).
        cache_on = os.environ.get("EXTMCMC_DATA_CACHE", "1") != "0"
        slots = 3.0 if cache_on else 10.0
        n_obs, flops_per_iter, sweeps_per_iter = G * ng, 2.0 * slots * C * G * ng, 1 if cache_on else 4
        desc = (f"BASELINE cfg4: hierarchical normal, {G} groups x {ng} obs, {C} chains/GPU, "
                "schedule MALA(theta_1..8) + RW(mu) + RW-pos(tau), full 10 x 10 running covariance; "
                + ("data-sum cache on: the sums over the observations are recomputed only when theta_1..8 move "
                   "(1 sweep per iteration)" if cache_on else "data-sum cache off: every element sweeps (4 per iteration)"))
    NUc = len(ups)
    # iterations per extmcmc_run_block: cfg 4 runs blocks of 10 iterations (30 schedule elements, like the
    # cfg 5 sub-record and well below run_()'s default block of 128 elements) -- the last element of a block
    # cannot leave its bookkeeping to the next element's kernels, which costs ~4 us per block; cfg 3: 1
    IPB = CFG4_BLOCK_ITERS if workload == "cfg4" else 1

    def make(instrument):
        mcmc = em.MCMC(ups, backend=em.CUDAMCMCBackend(n_chains=C, device=local, seed=7, history="none", block_len=NUc * IPB,
                                                       use_graphs=not instrument, instrument=instrument,
                                                       chain_offset=chain_offset))
        init_(mcmc, 1, data, th0)
        return mcmc.workspace
    up = lambda n: -(-n // IPB) * IPB            # whole blocks
    K, Wm = steps, up(3)                         # main() admits only whole blocks of timed steps
    ws = make(False)
    sampler = ClockSampler(local)
    _generic_timed(ws, _abi, NUc, 0, Wm, ipb=IPB)
    sampler.start()
    l0 = ws.lib.extmcmc_launch_count(ws.handle)
    ms_total = _generic_timed(ws, _abi, NUc, K, 0, it0=Wm + 1, ipb=IPB)
    launches = int(ws.lib.extmcmc_launch_count(ws.handle) - l0)
    ext = [Wm + 1 + K]

    def hold():
        _generic_timed(ws, _abi, NUc, up(5), 0, it0=ext[0], ipb=IPB); ext[0] += up(5)
    clocks = sampler.stop(extend=hold)
    variant = ws.lib.extmcmc_sweep_variant_name(ws.handle).decode()
    pk64, lanes = fp64_peaks(ws, clocks)
    pkmma = ctypes.c_double()
    ws._ck(ws.lib.extmcmc_measure_dmma_peak(ws.handle, ctypes.byref(pkmma)))
    acc = ws.stats()["n_accept"].sum(axis=1) / np.maximum(ws.stats()["n_prop"].sum(axis=1), 1)
    ws.close()
    wi = make(True)
    _generic_timed(wi, _abi, NUc, 0, Wm, ipb=IPB)
    msw, nl = ctypes.c_float(), ctypes.c_int64()
    wi._ck(wi.lib.extmcmc_get_sweep_time(wi.handle, ctypes.byref(msw), ctypes.byref(nl)))
    step_ms = _generic_timed(wi, _abi, NUc, min(K, 20), 0, it0=Wm + 1, ipb=IPB)
    wi._ck(wi.lib.extmcmc_get_sweep_time(wi.handle, ctypes.byref(msw), ctypes.byref(nl)))
    kern_ms = msw.value / max(nl.value, 1)
    wi.close()
    launches_per_iter = nl.value / float(min(K, 20))
    peak = max(pkmma.value, pk64, lanes) if workload == "cfg3" else max(pk64, lanes)
    ach = flops_per_iter / launches_per_iter / (kern_ms * 1e-3) / 1e12
    return {
        "workload": desc, "ms_per_step": ms_total / K, "steps": K,
        "block": f"{IPB} iteration(s) ({IPB * NUc} schedule elements) per extmcmc_run_block, one CUDA event pair per block",
        "value": float(C) * K * NUc * n_obs / (ms_total * 1e-3), "unit": "chain-step*obs/s",
        "roofline": {"kernel": variant, "bound": "tensor" if workload == "cfg3" else "fp64",
                     "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if peak else None,
                     "peak_source": "largest of: FP64 DMMA / FMA micro-benchmarks in this process, SMs x 64 lanes x 2 x SM clock under load",
                     "fp64_fma_probe": pk64, "fp64_dmma_probe": pkmma.value, "peak_lanes_x_clock": lanes,
                     "avg_launch_ms": kern_ms, "launches_timed": int(nl.value),
                     "launches_per_iteration": launches_per_iter, "sweeps_per_iteration": sweeps_per_iter,
                     "share_of_step": msw.value / step_ms if step_ms else None,
                     "algorithmic_flops_per_iteration": flops_per_iter,
                     "floor_ms_per_iteration": flops_per_iter / (peak * 1e12) * 1e3 if peak else None,
                     "traffic": None, "traffic_source": "not captured (the data set is L2 / shared-memory resident)" if workload == "cfg4"
                     else "see profiles/ (ncu --set full of the logistic sweep)"},
        "accept_rate_per_update": [float(a) for a in acc], "gpu_launches": launches, "clocks": clocks}


def run_ours(args):
    import ctypes
    import torch
    import extensiblemcmc_jl_b200 as em
    from extensiblemcmc_jl_b200 import _abi, parallel as par

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the GPU path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    K, Wm = args.steps, max(args.warmup, 3)
    C = CHAINS_PER_GPU
    x = cfg2_data()
    peaks, peak_src = measured_peaks()

    # ---- value: device-resident, one CUDA graph per iteration, L2 flushed between steps ------------
    ws = make_ws(em, x, C, rank * C, local, block_len=NU, use_graphs=True)
    variant = ws.lib.extmcmc_sweep_variant_name(ws.handle).decode()
    sampler = ClockSampler(local)
    barrier()
    timed_steps(ws, _abi, C, 0, Wm)                # warm-up (first launches, clocks)
    l1 = ws.lib.extmcmc_launch_count(ws.handle)
    sampler.start()
    barrier()
    ms_total = timed_steps(ws, _abi, C, K, 0, it0=Wm + 1)
    barrier()
    if args.dump_outputs:   # read back before the untimed continuation below moves the chains on
        dump_outputs(args.dump_outputs, last_step_outputs(ws, _abi, Wm + K), dist)
    ext = [Wm + 1 + K]   # a timed region shorter than three samples: keep the same load going, untimed

    def hold():
        timed_steps(ws, _abi, C, 20, 0, it0=ext[0]); ext[0] += 20
    clocks = sampler.stop(extend=hold)
    # kernels launched by the timed steps themselves (the untimed continuation above excluded)
    launches = int((ws.lib.extmcmc_launch_count(ws.handle) - l1) * K / max(ext[0] - (Wm + 1), 1))
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    units = float(world) * C * K * NU * N_OBS
    value = units / (ms_total * 1e-3)
    fp64_probe, lanes_peak = fp64_peaks(ws, clocks)
    ws.close()

    # ---- roofline of the dominant kernel: every launch of it bracketed by events --------------
    wsi = make_ws(em, x, C, rank * C, local, block_len=NU, use_graphs=False, instrument=True)
    timed_steps(wsi, _abi, C, 0, Wm)
    msw, nl = ctypes.c_float(), ctypes.c_int64()
    wsi._ck(wsi.lib.extmcmc_get_sweep_time(wsi.handle, ctypes.byref(msw), ctypes.byref(nl)))
    n_instr = min(K, 50)
    step_ms_instr = timed_steps(wsi, _abi, C, n_instr, 0)
    wsi._ck(wsi.lib.extmcmc_get_sweep_time(wsi.handle, ctypes.byref(msw), ctypes.byref(nl)))
    kern_ms = msw.value / max(nl.value, 1)
    sweeps_per_launch = n_instr * NU / max(nl.value, 1)     # 1 for the per-step kernels; a block kernel runs several
    sweep_share = msw.value / step_ms_instr if step_ms_instr > 0 else None
    wsi.close()
    flops = 3.0 * C * N_OBS * sweeps_per_launch    # SURVEY 8(d): 1 SUB + 1 FMA per chain x observation
    ach_tf = flops / (kern_ms * 1e-3) / 1e12
    fp64_peak = max(fp64_probe, lanes_peak)
    traffic, traffic_src = ncu_traffic("sweep_gsn1d_chains_kernel", "ncu_full_chains_r02.csv")
    roofline = {
        "kernel": variant, "bound": "fp64", "achieved": ach_tf, "peak": fp64_peak,
        "unit": "TFLOP/s", "frac": ach_tf / fp64_peak if fp64_peak else None,
        "peak_source": "larger of the FP64 FMA micro-benchmark run in this process and SMs x 64 lanes x 2 flop x SM clock "
                       "sampled under load (MEASURED_PEAKS.json has no FP64 figure)",
        "fp64_fma_probe": fp64_probe, "peak_lanes_x_clock": lanes_peak,
        # 2 FP64 issue slots (DADD + DFMA) per chain x observation against 3 flop counted: the
        # formulation's ceiling is 0.75 of the FMA-rate peak; issue_frac is the fraction of that ceiling
        "issue_frac": (2.0 * C * N_OBS * sweeps_per_launch / (kern_ms * 1e-3)) / (fp64_peak * 1e12 / 2.0) if fp64_peak else None,
        "avg_launch_ms": kern_ms, "launches_timed": int(nl.value), "update_steps_per_launch": sweeps_per_launch,
        "share_of_step": sweep_share,
        "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": 8.0 * N_OBS,
        "traffic": traffic, "traffic_source": traffic_src,
        "hbm": {"achieved": 8.0 * N_OBS / (kern_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                "unit": "GB/s", "frac": 8.0 * N_OBS / (kern_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "peak_source": peak_src + " (MEASURED_PEAKS.json)" if peak_src == "measured" else "fallback"},
    }

    # ---- the HBM-bound regime of the same kernel family (cfg 5 shape on one GPU) ------------------
    roofline_hbm = None
    if rank == 0 and not args.skip_hbm:
        n5, c5 = 1 << 28, 8                       # 2 GiB of observations, 8 chains
        ups = cfg2_updates(em)
        from extensiblemcmc_jl_b200.mcmc import init_
        m5 = em.MCMC(ups, backend=em.CUDAMCMCBackend(n_chains=c5, device=local, seed=6, history="none",
                                                     block_len=NU, use_graphs=False, instrument=True, sweep_variant=2))
        init_(m5, 1, dict(P=em.GsnTargetLaw([0.0]), obs=em.DeviceGeneratedObs(n5, 1.5, 2.0, 6)),
              np.repeat(np.array([[1.5], [4.0]]), c5, axis=1))
        w5 = m5.workspace
        for _ in range(3):
            w5.eval_loglik()
        w5._ck(w5.lib.extmcmc_get_sweep_time(w5.handle, ctypes.byref(msw), ctypes.byref(nl)))
        for _ in range(10):
            w5.eval_loglik()
        w5._ck(w5.lib.extmcmc_get_sweep_time(w5.handle, ctypes.byref(msw), ctypes.byref(nl)))
        t5 = msw.value / max(nl.value, 1)
        gbs = 8.0 * n5 / (t5 * 1e-3) / 1e9
        tr5, tr5_src = ncu_traffic("sweep_gsn1d_obs_kernel", "ncu_full_obs_r02.csv")
        roofline_hbm = {"kernel": w5.lib.extmcmc_sweep_variant_name(w5.handle).decode(),
                        "workload": f"cfg5 shape on 1 GPU: C={c5}, N=2^28 (2 GiB > L2)", "bound": "hbm",
                        "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": gbs / peaks["hbm_gbs"], "avg_launch_ms": t5,
                        "peak_source": peak_src,
                        "traffic": tr5, "traffic_source": tr5_src, "algorithmic_bytes": 8.0 * n5}
        w5.close()

    # ---- e2e: the whole job through run_() with host buffers --------------------------------------
    M = args.e2e_iters
    th0 = cfg2_theta_init(x, C, rank * C)

    def job(m_iters):
        mcmc = em.MCMC(cfg2_updates(em), backend=em.CUDAMCMCBackend(
            n_chains=C, device=local, seed=3, chain_offset=rank * C, block_len=128))
        return em.run_(mcmc, m_iters, dict(P=em.GsnTargetLaw([0.0]), obs=x), th0)

    w_, _ = job(8); w_.close()                   # warm-up of the API path
    barrier()
    t0 = time.perf_counter()
    ws_e, lws_e = job(M)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    t = torch.tensor([wall], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall = float(t.item())
    e2e_value = float(world) * C * M * NU * N_OBS / wall
    h2d = (8.0 * N_OBS + 8.0 * 2 * C) / M
    d2h = NU * C * (2 * 2 * 8 + 2 * 8 + 1)
    ess_per_sec = None
    if rank == 0 and M >= 400:
        tr = ws_e.sub_ws.state_history[M // 2:, 1][:, :, ::8]      # post warm-up, every 8th chain
        ess = em.ess_geyer(tr).min(axis=0)                          # min over params, per chain
        ess_per_sec = float(ess.mean() * C * world / wall)
    acc_rate = float(np.mean([l.acceptance_history.mean() for l in lws_e]))
    ws_e.close()
    barrier()

    # ---- BASELINE cfg 3 / cfg 4 on one GPU (before cfg 5: its HBM-bound sweeps run the board into
    # its power limit, and a short cfg 4 run right after them is timed at a capped clock) -------------
    cfg3 = cfg4 = None
    if rank == 0 and world == 1 and not args.skip_extras:
        def guarded(fn):   # a failed sub-record is reported as such and never costs the headline line
            try:
                return fn()
            except Exception as e:
                return {"error": repr(e)}
        cfg4 = guarded(lambda: measure_cfg34(args, "cfg4", em, _abi, local, args.cfg4_steps))
        if "EXTMCMC_DATA_CACHE" not in os.environ and "error" not in cfg4:
            # the same workload with every element streaming the observations (round-1 / early round-2 path)
            os.environ["EXTMCMC_DATA_CACHE"] = "0"
            try:
                off = guarded(lambda: measure_cfg34(args, "cfg4", em, _abi, local, args.cfg4_steps))
            finally:
                del os.environ["EXTMCMC_DATA_CACHE"]
            cfg4["without_data_cache"] = {k: off[k] for k in ("workload", "ms_per_step", "block", "value", "unit", "roofline", "gpu_launches", "error")
                                          if k in off}
        cfg3 = guarded(lambda: measure_cfg34(args, "cfg3", em, _abi, local, args.cfg3_steps))
    elif world > 1 and not args.skip_extras:
        # BASELINE cfg 4 as it is stated: 8192 chains per GPU (65536 over 8 GPUs), chains sharded, no
        # collective.  Every rank runs its own shard at the same time; the time is the max over ranks.
        barrier()
        try:
            rec = measure_cfg34(args, "cfg4", em, _abi, local, args.cfg4_steps, chain_offset=rank * 8192)
        except Exception as e:   # a failed sub-record must not take the collective (and the headline) down
            rec = {"error": repr(e), "ms_per_step": float("inf")}
        t = torch.tensor([rec["ms_per_step"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0 and not np.isfinite(t.item()):
            cfg4 = {"error": rec.get("error", "the sub-record failed on another rank")}
        elif rank == 0:
            per_gpu = rec["value"] * rec["ms_per_step"] / t.item()
            cfg4 = dict(rec, ms_per_step=t.item(), value=per_gpu * world, n_gpus=world, chains_total=8192 * world,
                        timing="every rank times its own shard with CUDA events; max over ranks",
                        roofline_of="rank 0")

    # ---- BASELINE cfg 5 (observations sharded, strong scaling, cross-rank exchange) ----------------
    strong_cfg5 = None
    if not args.skip_cfg5:
        strong_cfg5 = measure_cfg5(args, em, _abi, par, dist, rank, world, local, peaks, peak_src)

    # ---- CPU baseline: the oracle (a port of the reference's algorithm), 1 core -------------------
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        cpu = cpu_oracle_rate(x, n_chains=8, n_iters=args.cpu_iters, n_threads=1)
        cpu["sample"] = (f"{cpu.pop('chains')} chains x {cpu.pop('iters')} iterations of cfg2 "
                         f"(N=1e6, 2 updates), single thread, oracle = CPU restatement of "
                         f"ExtensibleMCMC.jl's algorithm (Julia unavailable)")

    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    out = {
        "metric": "chain-steps x obs/sec", "value": value, "unit": "chain-step*obs/s",
        "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms_total / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "BASELINE cfg2: 4096 chains/GPU x iid Gaussian likelihood, N=1e6 obs, "
                               "2 adaptive uniform random-walk updates per iteration",
                   "chains_per_gpu": C, "n_obs": N_OBS, "updates_per_step": NU,
                   "parallelism": f"chains sharded over {world} GPU(s), observations replicated, no collective",
                   "l2": "flushed (320 MiB write, untimed) before every timed step",
                   "timing": "one CUDA event pair per step on the library stream, no host sync inside the loop, summed; max over ranks"},
        "roofline": roofline, "roofline_hbm": roofline_hbm, "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "chain-step*obs/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "iters": M, "wall_s": wall,
                "what": "run_(mcmc, M, data, theta0): obs upload + all blocks + every history row copied to host"},
        "ess_per_sec": ess_per_sec, "accept_rate": acc_rate,
        "gpu_launches": launches, "clocks": clocks,
        "strong_cfg5": strong_cfg5, "cfg3": cfg3, "cfg4": cfg4,
    }
    print(json.dumps(out))


def _generic_timed(ws, _abi, n_updates, K, W, it0=1, ipb=1):
    """W warm-up + K timed MCMC iterations of an n_updates-element schedule, `ipb` iterations per
    extmcmc_run_block (one CUDA event pair per block; K and W are rounded up to whole blocks by the
    caller).  Returns the summed milliseconds of the K timed iterations."""
    import ctypes
    lib, h = ws.lib, ws.handle
    assert K % ipb == 0 and W % ipb == 0

    def block(it):
        arr = (_abi.Step * (n_updates * ipb))()
        for i in range(ipb):
            for pj in range(n_updates):
                e = arr[i * n_updates + pj]
                first = it + i == 1 and pj == 0
                e.mcmciter, e.pidx = it + i, pj
                e.prev_pidx = -1 if first else (pj - 1 if pj else n_updates - 1)
                e.prev_mcmciter = 0 if first else (it + i if pj else it + i - 1)
        return arr
    it = it0
    for _ in range(W // ipb):
        ws._ck(lib.extmcmc_run_block(h, block(it), n_updates * ipb)); it += ipb
    ws.sync()
    K = K // ipb
    for k in range(K):
        ws._ck(lib.extmcmc_event_record(h, 2 * k))
        ws._ck(lib.extmcmc_run_block(h, block(it), n_updates * ipb)); it += ipb
        ws._ck(lib.extmcmc_event_record(h, 2 * k + 1))
    ws.sync()
    ms, total = ctypes.c_float(), 0.0
    for k in range(K):
        ws._ck(lib.extmcmc_event_elapsed(h, 2 * k, 2 * k + 1, ctypes.byref(ms)))
        total += ms.value
    return total


def run_secondary(args):
    """Stand-alone runs of the secondary workloads (`--workload cfg3|cfg4|cfg5`): the same
    measurements the default run attaches as sub-records, printed as one JSON line."""
    import torch
    import extensiblemcmc_jl_b200 as em
    from extensiblemcmc_jl_b200 import _abi, parallel as par
    rank, world, local = par.env_rank_world()
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks, peak_src = measured_peaks()
    if args.workload == "cfg5":
        rec = measure_cfg5(args, em, _abi, par, dist, rank, world, local, peaks, peak_src)
    else:
        if world > 1:
            raise SystemExit("cfg3 / cfg4 shard by chains (no collective): run them on one GPU, or the default bench for scaling")
        rec = measure_cfg34(args, args.workload, em, _abi, local, args.steps)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        rec["n_gpus"] = world
        print(json.dumps(rec))


def cpu_oracle_rate(x, n_chains, n_iters, n_threads):
    import extensiblemcmc_jl_b200 as em
    from oracle import oracle as orc
    ups = cfg2_updates(em)
    o = orc.Oracle(em.GsnTargetLaw([0.0]), ups, x, cfg2_theta_init(x, n_chains), n_chains, seed=3)
    steps = list(em.MCMCSchedule(n_iters, NU))
    t0 = time.perf_counter()
    o.run(steps, n_threads=n_threads, record=False)
    dt = time.perf_counter() - t0
    return {"value": n_chains * n_iters * NU * float(len(x)) / dt, "unit": "chain-step*obs/s",
            "cores": n_threads, "kind": "port", "chains": n_chains, "iters": n_iters, "wall_s": dt}


def run_reference(args):
    """Reference arm: the reference's own CPU algorithm (oracle port; Julia is not in the
    image) on all host threads, bounded sample of the same workload per step."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import extensiblemcmc_jl_b200 as em
    from oracle import oracle as orc
    nthr = os.cpu_count() or 1
    x = cfg2_data()
    n_chains = 8 * nthr                       # per step: 8 chains per thread x 1 iteration x N=1e6
    ups = cfg2_updates(em)
    o = orc.Oracle(em.GsnTargetLaw([0.0]), ups, x, cfg2_theta_init(x, n_chains), n_chains, seed=3)
    K, Wm = args.steps, max(args.warmup, 1)
    sched = list(em.MCMCSchedule(Wm + K, NU))
    o.run(sched[:Wm * NU], n_threads=nthr, record=False)
    t0 = time.perf_counter()
    o.run(sched[Wm * NU:], n_threads=nthr, record=False)
    dt = time.perf_counter() - t0
    value = n_chains * K * NU * float(N_OBS) / dt
    sample = (f"{n_chains} chains x 1 iteration of cfg2 (N=1e6, 2 updates) per step, {K} steps, "
              f"{nthr} threads; oracle = CPU restatement of ExtensibleMCMC.jl's algorithm (Julia unavailable)")
    # ESS/s (BASELINE.json's second metric): effective samples per chain-iteration from a full-length
    # cfg2 trace of one chain per thread (M iterations, second half kept, Geyer estimator, minimum
    # over the parameters -- the same definition as the GPU arm) x the chain-iterations/s timed above
    ess_per_sec = ess_note = None
    if not args.skip_ess:
        M = args.ref_ess_iters
        oe = orc.Oracle(em.GsnTargetLaw([0.0]), cfg2_updates(em), x, cfg2_theta_init(x, nthr), nthr, seed=3)
        te = time.perf_counter()
        re_ = oe.run(list(em.MCMCSchedule(M, NU)), n_threads=nthr, record=False)
        te = time.perf_counter() - te
        tr = re_["theta"].reshape(M, NU, 2, nthr)[M // 2:, 1]
        ess_iter = float(em.ess_geyer(tr).min(axis=0).mean() / (M - M // 2))
        ess_per_sec = ess_iter * (n_chains * K / dt)
        ess_note = (f"ESS per chain-iteration {ess_iter:.4g} from {nthr} chains x {M} iterations of cfg2 "
                    f"(second half; {te:.1f} s of CPU time, untimed) x chain-iterations/s of the timed steps")
    print(json.dumps({
        "impl": "reference", "metric": "chain-steps x obs/sec", "value": value, "unit": "chain-step*obs/s",
        "n_gpus": args.gpus, "steps": K, "warmup": Wm, "ms_per_step": dt / K * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "BASELINE cfg2 (bounded sample): iid Gaussian likelihood, N=1e6 obs, "
                               "2 adaptive uniform random-walk updates per iteration", "n_obs": N_OBS},
        "cpu_baseline": {"value": value, "unit": "chain-step*obs/s", "cores": nthr, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "chain-step*obs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ess_per_sec": ess_per_sec, "ess_note": ess_note,
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-iters", type=int, default=2000, help="iterations of the end-to-end job (BASELINE cfg2: 2000)")
    ap.add_argument("--cpu-iters", type=int, default=600, help="iterations of the single-core CPU baseline (~10 s)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-hbm", action="store_true")
    ap.add_argument("--skip-cfg5", action="store_true", help="no strong_cfg5 sub-record")
    ap.add_argument("--skip-extras", action="store_true", help="no cfg3 / cfg4 sub-records (cfg3: N = 1 only; cfg4: every N, 8192 chains per GPU)")
    ap.add_argument("--skip-ess", action="store_true", help="reference arm: no ESS/s trace")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--cfg5-n-obs", type=int, default=1_000_000_000, help="cfg5: total observations over all ranks")
    ap.add_argument("--cfg5-iters", type=int, default=300, help="cfg5: timed MCMC iterations per exchange mode")
    ap.add_argument("--cfg3-n-obs", type=int, default=1_000_000)
    ap.add_argument("--cfg3-steps", type=int, default=5)
    ap.add_argument("--cfg4-steps", type=int, default=400)
    ap.add_argument("--ref-ess-iters", type=int, default=2000, help="reference arm: iterations of the ESS trace")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="cfg2: after the timed steps, write what the last one computed (chain state, log-likelihoods, "
                         "proposals, decisions, step sizes, chain statistics) as DIR/<name>.npy, float64; the inputs are "
                         "seeded, so two builds run with the same arguments can be compared array for array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.cfg4_steps % CFG4_BLOCK_ITERS or (args.workload == "cfg4" and args.steps % CFG4_BLOCK_ITERS):
        ap.error(f"cfg4 is timed in whole blocks of {CFG4_BLOCK_ITERS} iterations: its steps must be a multiple of that")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "cfg2"):
        ap.error("--dump-outputs writes the outputs of the cfg2 timed path (--impl ours, --workload cfg2)")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload != "cfg2":
        run_secondary(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
