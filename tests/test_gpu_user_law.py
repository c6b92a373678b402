"""User-defined device laws (DeviceLaw, EXTMCMC_LAW_USER) on the B200: the run-time compiled sweep
against numpy fp64 closed forms and finite differences, replay parity against the oracle's built-in
laws, the same decisions as the built-in GSN_IID_1D law under the own Philox stream, a conjugate
posterior, bit-identical launch variants, checkpoint / resume and the error paths."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from oracle import oracle as orc
from tests import user_laws as ul
from tests.parity import GpuSession, cfg2_updates, compare_histories, theta_init_for

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _session(src, grad, P, D, updates, X, th0, Cn, seed=0, **cfg):
    """GpuSession of a DeviceLaw: the library handle gets the law after creation."""
    law = em.DeviceLaw(src, P, D, gradient=grad)
    g = GpuSession(law, updates, X, th0, Cn, seed=seed, **cfg)
    g.ck(g.lib.extmcmc_set_user_law(g.h, src.encode(), 1 if grad else 0))
    return g


def _data(law, N, D, seed=0):
    rng = np.random.default_rng(seed)
    if law == "gsn1d":
        X = (1.5 + 2.0 * rng.standard_normal((N, 1)))
    else:
        P = D - 1 if law == "logistic" else D
        nx = P if law == "logistic" else P - 1
        X = np.empty((N, D))
        X[:, :nx] = rng.standard_normal((N, nx)) / math.sqrt(max(nx, 1))
        beta = 0.5 * rng.standard_normal(P)
        if law == "logistic":
            X[:, nx] = rng.random(N) < 1.0 / (1.0 + np.exp(-X[:, :nx] @ beta))
        else:
            X[:, nx] = rng.poisson(np.exp(beta[0] + X[:, :nx] @ beta[1:]))
    return X


def _theta(law, P, Cn, seed=1):
    rng = np.random.default_rng(seed)
    if law == "gsn1d":
        return np.stack([1.5 + 0.1 * rng.standard_normal(Cn), 4.0 * np.exp(0.1 * rng.standard_normal(Cn))])
    return 0.3 * rng.standard_normal((P, Cn))


def _reference(law, th, X):
    t, g = ul.LAWS[law][2](th, X)
    return t.sum(axis=0), np.abs(t).sum(axis=0), g.sum(axis=1), np.abs(g).sum(axis=1)


SHAPES = [("gsn1d", 1, 1, 1), ("gsn1d", 7, 5, 1), ("gsn1d", 1000, 4096, 1), ("gsn1d", 2**20 + 3, 33, 1),
          ("logistic", 1000, 33, 8), ("logistic", 7, 4096, 3), ("logistic", 2**20 + 3, 5, 8), ("logistic", 1, 1, 3),
          ("poisson_reg", 1000, 5, 8), ("poisson_reg", 7, 33, 3), ("poisson_reg", 2**20 + 3, 1, 1),
          ("poisson_reg", 1000, 4096, 3)]


@pytest.mark.parametrize("law,N,Cn,D", SHAPES)
def test_loglik_and_gradient_against_numpy(law, N, Cn, D):
    src, Pf, _ = ul.LAWS[law]
    P = Pf(D)
    X = _data(law, N, D)
    th = _theta(law, P, Cn)
    g = _session(src, True, P, D, [em.MALAUpdate(0.01, list(range(1, P + 1)))], X, th, Cn)
    assert g.variant() == "user_lanes" if Cn <= 32 else g.variant().startswith("user_chains_R")
    ll, gr = g.eval_grad()
    ll2 = g.eval_loglik()
    sub = np.unique(np.linspace(0, Cn - 1, min(Cn, 6)).astype(int))
    llw, lla, grw, gra = _reference(law, th[:, sub], X)
    assert np.all(np.abs(ll[sub] - llw) <= 1e-12 * lla), (ll[sub], llw)
    assert np.array_equal(ll, ll2)
    assert np.all(np.abs(gr[:, sub] - grw) <= 1e-10 * np.maximum(gra, 1e-300)), (gr[:, sub], grw)
    # central finite differences of the device's own log-likelihood
    c = int(sub[-1])
    for k in range(P):
        h = 1e-6 * max(1.0, abs(th[k, c]))
        fd = []
        for s in (+1, -1):
            t2 = th.copy()
            t2[k, c] += s * h
            g.ck(g.lib.extmcmc_set_state(g.h, _abi.dptr(np.ascontiguousarray(t2))))
            fd.append(g.eval_loglik()[c])
        assert abs((fd[0] - fd[1]) / (2 * h) - gr[k, c]) <= 1e-5 * max(1.0, gra[k, -1], abs(gr[k, c])), (k, fd, gr[k, c])
    g.close()


def _replay(builtin_law, src, grad, updates, X, Xu, y, th0, Cn, n_iters, seed, block=None, **cfg):
    """replay_compare with the oracle on the built-in law and the GPU on its DeviceLaw restatement."""
    steps = list(em.MCMCSchedule(n_iters, len(updates)))
    o = orc.Oracle(builtin_law, updates, X, th0, Cn, seed=seed, y=y)
    ro = o.run(steps, n_threads=8)
    g = _session(src, grad, builtin_law.n_params, Xu.shape[1], updates, Xu, th0, Cn, seed=seed,
                 n_steps_hint=len(steps), **cfg)
    block = block or len(steps)
    parts = [g.run(steps[b:b + block], replay=(ro["proposals"][b:b + block], ro["exp_draws"][b:b + block]))
             for b in range(0, len(steps), block)]
    rg = {k: np.concatenate([q[k] for q in parts]) for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted")}
    rep = compare_histories(ro, rg)
    rep["variant"] = g.variant()
    if rep["chains_diverged"] == 0:
        so, sg = o.stats(), g.stats()
        rep["eps_bitexact"] = all(np.array_equal(o.eps(u), g.eps(u)) for u in range(1, len(updates) + 1))
        rep["moments_bitexact"] = bool(np.array_equal(so["mean"], sg["mean"]) and np.array_equal(so["cov"], sg["cov"]))
        rep["rolling_ar_bitexact"] = bool(np.array_equal(so["rolling_ar"], sg["rolling_ar"]))
        rep["counts_equal"] = bool(np.array_equal(so["n_accept"], sg["n_accept"]))
    g.close()
    return rep


@pytest.mark.parametrize("Cn", [64, 640])
def test_replay_parity_gsn1d_restatement(Cn):
    rng = np.random.default_rng(0)
    x = 1.5 + 2.0 * rng.standard_normal(20000)
    rep = _replay(em.GsnTargetLaw([0.0], [[1.0]]), ul.GSN1D, False, cfg2_updates(eps0=0.05, scale=5e-3, k=10, offset=2.0),
                  x, x[:, None], None, theta_init_for(x, Cn), Cn, 40, seed=11, block=17)
    print(rep)
    assert rep["accept_mismatch"] == 0 and rep["theta_bitexact"] and rep["ll_rel_err"] < 1e-10, rep
    if rep["chains_diverged"] == 0:
        assert rep["eps_bitexact"] and rep["moments_bitexact"] and rep["rolling_ar_bitexact"] and rep["counts_equal"], rep


def test_replay_parity_logistic_restatement_under_mala():
    d = 8
    X = _data("logistic", 3000, d + 1, seed=9)
    Cn = 96
    th0 = 0.01 * np.random.default_rng(2).standard_normal((d, Cn))
    ups = [em.MALAUpdate(0.15, list(range(1, d + 1)), prior=em.StandardPrior(em.Normal(0.0, 10.0)),
                         adpt=em.AdaptationMALA(adapt_every_k_steps=5, scale=0.01, offset=1.0))]
    rep = _replay(em.LogisticLaw(d), ul.LOGISTIC, True, ups, np.ascontiguousarray(X[:, :d]), X, X[:, d].copy(),
                  th0, Cn, 40, seed=3, block=13, history_window=32)
    print(rep)
    assert rep["accept_mismatch"] == 0 and rep["theta_bitexact"] and rep["ll_rel_err"] < 1e-10, rep
    if rep["chains_diverged"] == 0:
        assert rep["eps_bitexact"] and rep["moments_bitexact"] and rep["rolling_ar_bitexact"] and rep["counts_equal"], rep


def test_same_decisions_as_the_builtin_law_under_own_philox():
    rng = np.random.default_rng(5)
    x = 1.5 + 2.0 * rng.standard_normal(50000)
    Cn, M = 512, 60
    th0 = theta_init_for(x, Cn)
    steps = list(em.MCMCSchedule(M, 2))
    ups = cfg2_updates(eps0=0.05, scale=5e-3, k=10, offset=2.0)
    gb = GpuSession(em.GsnTargetLaw([0.0], [[1.0]]), ups, x, th0, Cn, seed=7, n_steps_hint=len(steps))
    rb = gb.run(steps)
    gu = _session(ul.GSN1D, False, 2, 1, ups, x[:, None], th0, Cn, seed=7, n_steps_hint=len(steps))
    ru = gu.run(steps)
    mism = rb["accepted"] != ru["accepted"]
    first = np.where(mism.any(axis=0), mism.argmax(axis=0), len(steps))
    near_ties = 0
    for c in np.nonzero(first < len(steps))[0]:
        s = first[c]
        # a near-tie: the two log-likelihood ratios differ only by rounding (the sums are associated differently)
        llr_b, llr_u = rb["ll_prop"][s, c] - rb["ll"][s, c], ru["ll_prop"][s, c] - ru["ll"][s, c]
        assert abs(llr_b - llr_u) <= 1e-10 * abs(rb["ll"][s, c]), (c, s, llr_b, llr_u)
        near_ties += 1
    print("near-ties:", near_ties, "of", Cn, "chains")
    ok = np.arange(len(steps))[:, None] < first[None, :]
    assert np.array_equal(rb["theta"][np.broadcast_to(ok[:, None], rb["theta"].shape)],
                          ru["theta"][np.broadcast_to(ok[:, None], ru["theta"].shape)])
    rel = np.abs(rb["ll_prop"] - ru["ll_prop"])[ok] / np.abs(rb["ll_prop"][ok])
    assert rel.max() < 1e-10
    assert near_ties <= Cn // 100
    gb.close(); gu.close()


def test_poisson_posterior_with_gamma_prior():
    rng = np.random.default_rng(3)
    N, a, b = 200, 3.0, 2.0
    y = rng.poisson(4.0, N).astype(np.float64)
    law = em.DeviceLaw(ul.POISSON_RATE, 1, 1)
    up = [em.RandomWalkUpdate(em.UniformRandomWalk([0.1], [True]), [1], prior=em.StandardPrior(em.Gamma(a, 1.0 / b)))]
    Cn, M, burn = 256, 4000, 500
    mcmc = em.MCMC(up, backend=em.CUDAMCMCBackend(n_chains=Cn, seed=3, block_len=200))
    ws, _ = em.run_(mcmc, M, dict(P=law, obs=y[:, None]), [4.0])
    tr = ws.sub_ws.state_history[burn:, 0, 0]            # [M - burn, C]
    shape, rate = a + y.sum(), b + N
    mean_w, var_w = shape / rate, shape / rate ** 2
    ess = em.ess_geyer(tr).sum()
    mcse_mean = math.sqrt(tr.var() / ess)
    mcse_var = math.sqrt(((tr - tr.mean()) ** 2).var() / ess)
    assert abs(tr.mean() - mean_w) < 3 * mcse_mean, (tr.mean(), mean_w, mcse_mean)
    assert abs(tr.var() - var_w) < 3 * mcse_var, (tr.var(), var_w, mcse_var)
    ws.close()


_JOB = r"""
import json, sys, numpy as np
sys.path.insert(0, '.')
import extensiblemcmc_jl_b200 as em
from tests import user_laws as ul
from tests.test_gpu_user_law import _session, _data
d = 8
X = _data("logistic", 5000, d + 1, seed=4)
th0 = 0.01 * np.random.default_rng(2).standard_normal((d, 300))
ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.02] * 4), [1, 2, 3, 4]),
       em.MALAUpdate(0.1, [5, 6, 7, 8], prior=em.StandardPrior(em.Normal(0.0, 10.0)),
                     adpt=em.AdaptationMALA(adapt_every_k_steps=5, scale=0.01, offset=1.0))]
steps = list(em.MCMCSchedule(12, 2))
out = {}
for name, cfg, block, splits in [("eager_all", dict(use_graphs=0), 24, [(0, 300)]),
                                 ("graph_all", dict(use_graphs=1), 24, [(0, 300)]),
                                 ("graph_b4", dict(use_graphs=1), 4, [(0, 300)]),
                                 ("eager_b1", dict(use_graphs=0), 1, [(0, 300)]),
                                 ("split", dict(use_graphs=1), 24, [(0, 130), (130, 300)])]:
    th, ll = [], []
    for lo, hi in splits:
        g = _session(ul.LOGISTIC, True, d, d + 1, ups, X, np.ascontiguousarray(th0[:, lo:hi]), hi - lo, seed=7,
                     chain_offset=lo, n_steps_hint=24, **cfg)
        for b in range(0, len(steps), block):
            g.run(steps[b:b + block])
        t, l = g.state()
        th.append(t); ll.append(l)
        g.close()
    out[name] = [np.concatenate(th, axis=1).tolist(), np.concatenate(ll).tolist()]
print(json.dumps(out))
"""


def test_launch_variants_are_bit_identical():
    res = []
    for env in ({}, {"EXTMCMC_LEAN": "0"}):
        e = dict(os.environ)
        e.update(env)
        r = subprocess.run([sys.executable, "-c", _JOB], capture_output=True, text=True, timeout=900, env=e, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-3000:]
        res.append(json.loads(r.stdout.strip().splitlines()[-1]))
    ref = res[0]["eager_all"]
    assert np.isfinite(np.array(ref[1])).all()
    for out in res:
        for name, v in out.items():
            assert v == ref, name


def test_checkpoint_resume_and_foreign_law():
    rng = np.random.default_rng(0)
    x = 1.5 + 2.0 * rng.standard_normal(30000)
    Cn, M = 200, 20
    th0 = theta_init_for(x, Cn)
    ups = cfg2_updates(eps0=0.05, scale=5e-3, k=5, offset=2.0)
    s1 = list(em.MCMCSchedule(M, 2))
    a = _session(ul.GSN1D, True, 2, 1, ups, x[:, None], th0, Cn, seed=5, n_steps_hint=2 * M)
    a.run(s1[:M]); a.run(s1[M:])
    th_a, ll_a = a.state()
    b = _session(ul.GSN1D, True, 2, 1, ups, x[:, None], th0, Cn, seed=5, n_steps_hint=2 * M)
    b.run(s1[:M])
    n = C.c_int64()
    b.ck(b.lib.extmcmc_checkpoint_size(b.h, C.byref(n)))
    blob = (C.c_uint8 * n.value)()
    b.ck(b.lib.extmcmc_checkpoint_save(b.h, blob, n.value))
    c = _session(ul.GSN1D, True, 2, 1, ups, x[:, None], th0 * 0 + th0[:, :1], Cn, seed=5, n_steps_hint=2 * M)
    c.ck(c.lib.extmcmc_checkpoint_load(c.h, blob, n.value))
    c.seq = M
    c.run(s1[M:])
    th_c, ll_c = c.state()
    assert np.array_equal(th_a, th_c) and np.array_equal(ll_a, ll_c)
    # the same shapes under another law source are refused
    other = ul.GSN1D.replace("g[1] +=", "g[1] += 0.0 +")
    d = _session(other, True, 2, 1, ups, x[:, None], th0, Cn, seed=5, n_steps_hint=2 * M)
    assert d.lib.extmcmc_checkpoint_load(d.h, blob, n.value) == _abi.EINVAL
    assert b"another user law" in d.lib.extmcmc_last_error(d.h)
    for s in (a, b, c, d):
        s.close()


def test_error_paths():
    rng = np.random.default_rng(1)
    x = 1.0 + rng.standard_normal(1000)
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([3.0]), [2])]   # steps the variance far below 0
    th0 = np.array([[1.0] * 64, [0.05] * 64])
    # domain violation: EDOMAIN at sync, the proposal is rejected, the state stays in the domain
    g = _session(ul.GSN1D, False, 2, 1, ups, x[:, None], th0, 64, seed=1, n_steps_hint=20)
    out = g.run(list(em.MCMCSchedule(20, 1)))
    assert out["rc"] == _abi.EDOMAIN
    bad = out["theta_prop"][:, 1] <= 0
    assert bad.any() and np.isnan(out["ll_prop"][bad]).all() and not out["accepted"][bad].any()
    assert (g.state()[0][1] > 0).all()
    g.close()
    # a run before extmcmc_set_user_law: EINVAL
    law = em.DeviceLaw(ul.GSN1D, 2, 1)
    g = GpuSession(law, ups, x[:, None], th0, 64, n_steps_hint=8)
    arr = orc.steps_array(list(em.MCMCSchedule(2, 1)))
    assert g.lib.extmcmc_run_block(g.h, arr, 2) == _abi.EINVAL
    assert g.lib.extmcmc_eval_loglik(g.h, _abi.dptr(np.empty(64))) == _abi.EINVAL
    # MALA and eval_grad on a law without gradient: EUNSUPPORTED
    g.ck(g.lib.extmcmc_set_user_law(g.h, ul.GSN1D.encode(), 0))
    assert g.lib.extmcmc_eval_grad(g.h, None, _abi.dptr(np.empty((2, 64)))) == _abi.EUNSUPPORTED
    u, _k = em.MALAUpdate(0.1, [1, 2]).to_abi(2)
    assert g.lib.extmcmc_set_update(g.h, 0, C.byref(u)) == _abi.EUNSUPPORTED
    g.close()
    with pytest.raises(_abi.ExtMCMCError) as ei:
        em.run_(em.MCMC([em.MALAUpdate(0.1, [1, 2])], backend=em.CUDAMCMCBackend(n_chains=8)), 5,
                dict(P=law, obs=x[:, None]), [1.0, 1.0])
    assert ei.value.code == _abi.EUNSUPPORTED
