"""Chunked forward-mode gradients of user-defined laws on the B200 (DeviceLaw(..., gradient="forward",
chunk=...), extmcmc_set_user_law_chunked): every chunk kernel under every mapping against the
extended-precision references of tests/user_laws_chunked.py, the same bits as the unchunked forward
sweep at every width on a pinned plan (gradients and MALA under replay), the posterior of a Gaussian
regression at P = 24, bit-identical launch variants, checkpoint / resume, the launch count and the
domain flag."""
import ctypes as C
import math

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws as ul
from tests import user_laws_chunked as uc
from tests import user_laws_forward as uf
from tests.parity import GpuSession
from tests.test_gpu_user_law_forward import G_TOL, HAND_TOL, _law_data, _law_theta

pytestmark = pytest.mark.gpu

N_ROWS = 3001
VARIANTS = [11, 12, 14, 2]      # forced chains R = 1 / 2 / 4 (as far as the budget allows) and lanes


def _session(src, P, D, updates, X, th0, Cn, chunk="auto", seed=0, **cfg):
    law = em.DeviceLaw(src, P, D, gradient="forward", chunk=chunk)
    g = GpuSession(law, updates, X, th0, Cn, seed=seed, **cfg)
    g.ck(law.abi_attach(g.lib, g.h))
    return g, law


def _ups():
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.01]), [1])]


def _reference(terms, th, X, chunk=16):
    Cn = th.shape[1]
    ll, gr, gra = np.empty(Cn), np.empty((th.shape[0], Cn)), np.empty((th.shape[0], Cn))
    for lo in range(0, Cn, chunk):
        t, g = terms(th[:, lo:lo + chunk], X, dtype=np.longdouble)
        ll[lo:lo + chunk] = t.sum(axis=0)
        gr[:, lo:lo + chunk] = g.sum(axis=1)
        gra[:, lo:lo + chunk] = np.abs(g).sum(axis=1)
    return ll, gr, gra


def _rmax(P, K):
    n = (P + 1) * (K + 1)
    return 4 if 4 * n <= 40 else 2 if 2 * n <= 40 else 1


# (law, P, chunk): the library's widths (20 = 4 x 5; ragged: 17 = 3 x 5 + 2, 24 = 4 x 5 + 4,
# 33 = 6 x 5 + 3, 64 = 12 x 5 + 4),
# every field live (pos_reg), the most chunks (64 at K = 4: 16), and P <= 16 at K = 1 (R up to 4)
CASES = [("poisson_reg", 20, "auto"), ("gauss_reg_scale", 17, "auto"), ("pos_reg", 24, "auto"),
         ("logistic", 33, "auto"), ("gauss_reg", 64, "auto"), ("poisson_reg", 64, 4), ("poisson_reg", 3, 1)]


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name,P,chunk", CASES)
def test_every_chunk_kernel_every_chain(name, P, chunk, variant):
    src, Df, terms = uc.LAWS[name]
    D, Cn = Df(P), 701
    X = uc.data(name, N_ROWS, P, seed=21)
    th = uc.theta(name, P, Cn, seed=22)
    g, law = _session(src, P, D, _ups(), X, th, Cn, chunk=chunk, sweep_variant=variant)
    v = g.variant()
    K = law.chunk
    assert v == ("user_lanes" if variant == 2 else f"user_chains_R{min(variant - 10, _rmax(P, K))}"), v
    ll_v = g.eval_loglik()
    ll_g, gr = g.eval_grad()
    assert g.lib.extmcmc_sync(g.h) == _abi.OK
    assert np.array_equal(ll_g, ll_v), np.abs(ll_g - ll_v).max()
    llw, grw, gra = _reference(terms, th, X)
    e_g = np.abs(gr - grw) / (G_TOL * np.maximum(gra, 1e-300))
    e_ll = np.abs(ll_v - llw) / (G_TOL * np.abs(llw).clip(1.0))
    print(f"{name} P={P} K={K} {v}: grad err / tol {e_g.max():.3g}, ll err / tol {e_ll.max():.3g}")
    assert e_g.max() <= 1, (np.unravel_index(np.argmax(e_g), e_g.shape), e_g.max())
    assert e_ll.max() <= 1, e_ll.max()
    g.close()


@pytest.mark.parametrize("variant", [11, 2])
def test_chunked_against_hand_gradient_p32(variant):
    P = D = 32
    Cn = 701
    X = _law_data("poisson_reg", N_ROWS, D, seed=31)
    th = _law_theta("poisson_reg", P, Cn, seed=32)
    g, law = _session(uf.POISSON_REG, P, D, _ups(), X, th, Cn, sweep_variant=variant)
    _, gr = g.eval_grad()
    g.close()
    h = GpuSession(em.DeviceLaw(ul.POISSON_REG, P, D, gradient=True), _ups(), X, th, Cn, sweep_variant=variant)
    h.ck(h.lib.extmcmc_set_user_law(h.h, ul.POISSON_REG.encode(), _abi.USER_GRAD_HAND))
    _, gr_h = h.eval_grad()
    h.close()
    _, _, gra = _reference(ul.poisson_reg_terms, th, X)
    e = np.abs(gr - gr_h) / (HAND_TOL * np.maximum(gra, 1e-300))
    print(f"P=32 K={law.chunk}: forward against hand-written, err / tol {e.max():.3g}")
    assert e.max() <= 1, e.max()


# ---- the same bits at every width -------------------------------------------------------------------
# chains R = 1 at C = 701 and 3001 rows: 6 chain groups, S = 11 segments (n_pairs / 128) whatever the
# occupancy of each width's kernels, so the plan is the same at every width

PINNED = dict(sweep_variant=11)


@pytest.mark.parametrize("name,D", [("gsn1d", 1), ("poisson_rate", 1), ("logistic", 4), ("poisson_reg", 8),
                                    ("poisson_reg", 16)])
def test_every_width_gives_the_unchunked_bits(name, D):
    src, _, Pf, _ = uf.LAWS[name]
    P = Pf(D)
    Cn = 701
    X = _law_data(name, N_ROWS, D, seed=41)
    th = _law_theta(name, P, Cn, seed=42)
    law = em.DeviceLaw(src, P, D, gradient="forward")
    g = GpuSession(law, _ups(), X, th, Cn, **PINNED)
    g.ck(law.abi_attach(g.lib, g.h))
    ll0, gr0 = g.eval_grad()
    g.close()
    for K in sorted({1, 2, 3, P} & set(range(1, P + 1))):
        s, _ = _session(src, P, D, _ups(), X, th, Cn, chunk=K, **PINNED)
        ll, gr = s.eval_grad()
        assert s.variant() == "user_chains_R1"
        s.close()
        assert np.array_equal(ll, ll0) and np.array_equal(gr, gr0), (name, K)


def test_mala_under_replay_is_bit_identical_across_widths():
    D = P = 8
    Cn, M, tau = 256, 120, 0.02
    X = _law_data("poisson_reg", 2000, D, seed=8)
    th0 = 0.3 * np.random.default_rng(9).standard_normal((P, Cn))
    ups = [em.MALAUpdate(tau, list(range(1, P + 1)))]
    steps = list(em.MCMCSchedule(M, 1))
    props = None
    exps = np.random.default_rng(10).exponential(size=(M, Cn))
    runs = {}
    for K in (None, 8, 3, 1):
        law = em.DeviceLaw(uf.POISSON_REG, P, D, gradient="forward", chunk=K)
        g = GpuSession(law, ups, X, th0, Cn, seed=4, n_steps_hint=M, **PINNED)
        g.ck(law.abi_attach(g.lib, g.h))
        if props is None:
            props = np.ascontiguousarray(g.run(steps)["theta_prop"])   # the unchunked run's own proposals
            g.close()
            g = GpuSession(law, ups, X, th0, Cn, seed=4, n_steps_hint=M, **PINNED)
            g.ck(law.abi_attach(g.lib, g.h))
        runs[K] = g.run(steps, replay=(props, exps))
        g.close()
    ref = runs[None]
    assert 0.2 < ref["accepted"][1:].mean() < 0.95, ref["accepted"].mean()
    for K in (8, 3, 1):
        r = runs[K]
        for key in ("theta", "ll", "accepted", "theta_prop", "ll_prop"):
            assert np.array_equal(r[key], ref[key], equal_nan=True), (K, key)


# ---- posterior ---------------------------------------------------------------------------------------

def test_mala_recovers_the_gaussian_regression_posterior_p24():
    # flat prior: the posterior is N(beta_hat, sigma^2 (A^T A)^-1), A = [1, x]
    P, N = 24, 400
    rng = np.random.default_rng(12)
    Xc = rng.standard_normal((N, P - 1))
    beta = rng.standard_normal(P)
    y = beta[0] + Xc @ beta[1:] + uc.SIGMA * rng.standard_normal(N)
    rows = np.concatenate([Xc, y[:, None]], axis=1)
    A = np.concatenate([np.ones((N, 1)), Xc], axis=1)
    cov = uc.SIGMA ** 2 * np.linalg.inv(A.T @ A)
    bhat = np.linalg.solve(A.T @ A, A.T @ y)
    law = em.DeviceLaw(uc.GAUSS_REG, P, P, gradient="forward", chunk="auto")
    assert law.chunk == 5
    Cn, M, burn = 256, 3000, 500
    up = [em.MALAUpdate(0.02, list(range(1, P + 1)))]
    mcmc = em.MCMC(up, backend=em.CUDAMCMCBackend(n_chains=Cn, seed=5, block_len=100))
    th0 = bhat + 0.02 * rng.standard_normal(P)
    ws, _ = em.run_(mcmc, M, dict(P=law, obs=rows), list(th0))
    hist = ws.sub_ws.state_history[burn:, 0]                     # [M - burn, P, C]
    acc = np.mean(np.diff(hist, axis=0) != 0)
    worst = 0.0
    for k in range(P):
        tr = hist[:, k]
        ess = em.ess_geyer(tr).sum()
        mcse_mean = math.sqrt(tr.var() / ess)
        mcse_var = math.sqrt(((tr - tr.mean()) ** 2).var() / ess)
        zm = abs(tr.mean() - bhat[k]) / mcse_mean
        zv = abs(tr.var() - cov[k, k]) / mcse_var
        worst = max(worst, zm, zv)
        assert zm < 3 and zv < 3, (k, tr.mean(), bhat[k], mcse_mean, tr.var(), cov[k, k], mcse_var)
    print(f"P=24 K={law.chunk}: move rate {acc:.3f}, worst |error| / mcse {worst:.3g}")
    ws.close()


# ---- determinism ------------------------------------------------------------------------------------

def _det_problem(P=20):
    X = _law_data("poisson_reg", 5000, P, seed=4)
    th0 = 0.01 * np.random.default_rng(2).standard_normal((P, 300))
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.02, 0.02]), [1, 2]),
           em.MALAUpdate(0.01, list(range(3, P + 1)), prior=em.StandardPrior(em.Normal(0.0, 10.0)),
                         adpt=em.AdaptationMALA(adapt_every_k_steps=5, scale=0.01, offset=1.0))]
    return P, X, th0, ups


def test_launch_variants_are_bit_identical():
    P, X, th0, ups = _det_problem()
    steps = list(em.MCMCSchedule(12, 2))
    out = {}
    for name, cfg, block, splits in [("eager_all", dict(use_graphs=0), 24, [(0, 300)]),
                                     ("graph_all", dict(use_graphs=1), 24, [(0, 300)]),
                                     ("graph_b4", dict(use_graphs=1), 4, [(0, 300)]),
                                     ("eager_b1", dict(use_graphs=0), 1, [(0, 300)]),
                                     ("split", dict(use_graphs=1), 24, [(0, 130), (130, 300)])]:
        th, ll = [], []
        for lo, hi in splits:
            g, _ = _session(uf.POISSON_REG, P, P, ups, X, np.ascontiguousarray(th0[:, lo:hi]), hi - lo, seed=7,
                            chain_offset=lo, n_steps_hint=24, **cfg)
            for b in range(0, len(steps), block):
                g.run(steps[b:b + block])
            t, l = g.state()
            th.append(t)
            ll.append(l)
            g.close()
        out[name] = (np.concatenate(th, axis=1), np.concatenate(ll))
    ref = out["eager_all"]
    assert np.isfinite(ref[1]).all()
    assert not np.array_equal(ref[0], th0)
    for name, (t, l) in out.items():
        assert np.array_equal(t, ref[0]) and np.array_equal(l, ref[1]), name


def test_checkpoint_resume_p32_and_another_width_is_refused():
    P, X, th0, ups = _det_problem(32)
    Cn, M = 300, 20
    s1 = list(em.MCMCSchedule(M, 2))
    a, law = _session(uf.POISSON_REG, P, P, ups, X, th0, Cn, seed=5, n_steps_hint=2 * M)
    a.run(s1[:M]); a.run(s1[M:])
    th_a, ll_a = a.state()
    b, _ = _session(uf.POISSON_REG, P, P, ups, X, th0, Cn, seed=5, n_steps_hint=2 * M)
    b.run(s1[:M])
    n = C.c_int64()
    b.ck(b.lib.extmcmc_checkpoint_size(b.h, C.byref(n)))
    blob = (C.c_uint8 * n.value)()
    b.ck(b.lib.extmcmc_checkpoint_save(b.h, blob, n.value))
    c, _ = _session(uf.POISSON_REG, P, P, ups, X, th0 * 0 + th0[:, :1], Cn, seed=5, n_steps_hint=2 * M)
    c.ck(c.lib.extmcmc_checkpoint_load(c.h, blob, n.value))
    c.seq = M
    c.run(s1[M:])
    th_c, ll_c = c.state()
    assert np.array_equal(th_a, th_c) and np.array_equal(ll_a, ll_c)
    # the same source compiled at another width is another program: its blob is refused
    assert law.chunk != 8
    d, _ = _session(uf.POISSON_REG, P, P, ups, X, th0, Cn, chunk=8, seed=5, n_steps_hint=2 * M)
    assert d.lib.extmcmc_checkpoint_load(d.h, blob, n.value) == _abi.EINVAL
    for s in (a, b, c, d):
        s.close()


def test_unchunked_width_shares_checkpoints_with_the_forward_entry_point():
    D = P = 4
    X = _law_data("poisson_reg", 1000, D, seed=3)
    th0 = 0.01 * np.random.default_rng(2).standard_normal((P, 64))
    ups = [em.MALAUpdate(0.01, [1, 2, 3, 4])]
    a = GpuSession(em.DeviceLaw(uf.POISSON_REG, P, D, gradient="forward"), ups, X, th0, 64, seed=5)
    a.ck(a.lib.extmcmc_set_user_law(a.h, uf.POISSON_REG.encode(), _abi.USER_GRAD_FORWARD))
    a.run(list(em.MCMCSchedule(5, 1)))
    n = C.c_int64()
    a.ck(a.lib.extmcmc_checkpoint_size(a.h, C.byref(n)))
    blob = (C.c_uint8 * n.value)()
    a.ck(a.lib.extmcmc_checkpoint_save(a.h, blob, n.value))
    b, _ = _session(uf.POISSON_REG, P, D, ups, X, th0, 64, chunk=P, seed=5)
    b.ck(b.lib.extmcmc_checkpoint_load(b.h, blob, n.value))
    c, _ = _session(uf.POISSON_REG, P, D, ups, X, th0, 64, chunk=2, seed=5)
    assert c.lib.extmcmc_checkpoint_load(c.h, blob, n.value) == _abi.EINVAL
    for s in (a, b, c):
        s.close()


# ---- launches and the domain flag -------------------------------------------------------------------

@pytest.mark.parametrize("P,chunk,nc", [(17, "auto", 4), (64, "auto", 13), (64, 4, 16), (8, None, 1), (8, 3, 3)])
def test_launch_count_per_gradient_sweep(P, chunk, nc):
    X = _law_data("poisson_reg", 1000, P, seed=1)
    g, law = _session(uf.POISSON_REG, P, P, _ups(), X, np.zeros(P), 64, chunk=chunk)
    g.eval_loglik()
    n0 = g.lib.extmcmc_launch_count(g.h)
    g.eval_grad()
    n1 = g.lib.extmcmc_launch_count(g.h)
    g.eval_loglik()
    n2 = g.lib.extmcmc_launch_count(g.h)
    assert (n1 - n0, n2 - n1) == (nc + 1, 2), (law.chunk, n1 - n0, n2 - n1)
    g.close()


def test_failing_set_parameters_gives_nan_and_edomain():
    name, P = "gauss_reg_scale", 20
    src, Df, _ = uc.LAWS[name]
    Cn = 300
    X = uc.data(name, 1000, P, seed=2)
    th = uc.theta(name, P, Cn, seed=3)
    bad = np.zeros(Cn, bool)
    bad[::7] = True
    th[P - 1, bad] = -0.5
    g, law = _session(src, P, Df(P), _ups(), X, th, Cn)
    assert law.chunk == 5
    ll, gr = np.empty(Cn), np.empty((P, Cn))
    rc = g.lib.extmcmc_eval_grad(g.h, _abi.dptr(ll), _abi.dptr(gr))
    rc_sync = g.lib.extmcmc_sync(g.h)
    assert _abi.EDOMAIN in (rc, rc_sync), (rc, rc_sync)
    assert np.isnan(ll[bad]).all() and np.isnan(gr[:, bad]).all()
    assert np.isfinite(ll[~bad]).all() and np.isfinite(gr[:, ~bad]).all()
    g.close()
