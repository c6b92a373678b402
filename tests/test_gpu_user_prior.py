"""User-defined priors (DevicePrior) on a B200: restatements of the built-in priors give the built-in
prior's bits under the library's own Philox stream (histories, proposals, log-likelihoods, step sizes,
Sigma_B, running moments, state) for every random walk and MALA, on the built-in laws (GsnTargetLaw
d = 1 and 2) and a DeviceLaw; lp and grad lp of non-linear priors match 50-digit arithmetic; the redraw
loop runs in the prior's kernel; a Laplace prior's posterior matches quadrature; graphs, block
lengths, chain splits and checkpoints do not change the bits; the launch counts and refusals."""
import ctypes as C
import math

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws as ul
from tests import user_priors as up
from tests.parity import GpuSession, replay_compare

pytestmark = pytest.mark.gpu


def _session(law, ups, obs, th0, Cn, y=None, **cfg):
    g = GpuSession(law, ups, obs, th0, Cn, y=y, **cfg)
    if hasattr(law, "abi_attach"):
        g.ck(law.abi_attach(g.lib, g.h))
    for i, u in enumerate(ups):
        if hasattr(u.prior, "abi_attach"):
            g.ck(u.prior.abi_attach(g.lib, g.h, i))
    return g


def _run(law, ups, obs, th0, Cn, steps, block, y=None, **cfg):
    g = _session(law, ups, obs, th0, Cn, y=y, n_steps_hint=max(block, 1), **cfg)
    parts = [g.run(steps[b:b + block]) for b in range(0, len(steps), block)]
    out = {k: np.concatenate([q[k] for q in parts]) for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted")}
    out["rc"] = [q["rc"] for q in parts]
    # step sizes (uniform walk, MALA) and Sigma_B (mixture); a plain Gaussian walk keeps no per-chain state
    out["eps"] = [g.eps(u) for u in range(1, len(ups) + 1) if g.kernels[u - 1] != _abi.KERNEL_RW_GAUSS]
    out["haario"] = [np.concatenate(g.adapt_state(u)) for u in range(1, len(ups) + 1)
                     if isinstance(getattr(ups[u - 1], "adpt", None), em.HaarioTypeAdaptation)]
    out["stats"] = g.stats()
    out["state"] = g.state()
    out["launches"] = g.lib.extmcmc_launch_count(g.h)
    g.close()
    return out


def _assert_same(a, b):
    for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    # the same outcome per run (a Sigma_B that is not positive definite is EXTMCMC_EDOMAIN in both)
    assert set(a["rc"]) == set(b["rc"])
    for key in ("eps", "haario"):
        assert len(a[key]) == len(b[key]) and all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a[key], b[key]))
    for k, v in a["stats"].items():
        assert np.array_equal(v, b["stats"][k], equal_nan=True), k
    assert np.array_equal(a["state"][0], b["state"][0]) and np.array_equal(a["state"][1], b["state"][1], equal_nan=True)


# (builtin, restated) pairs on two coordinates
PRIORS = {
    "normal": (em.StandardPrior(em.Normal(0.5, 2.0)), (up.NORMAL, (0.5, 2.0))),
    "gamma": (em.StandardPrior(em.Gamma(2.0, 0.5)), (up.GAMMA, (2.0, 0.5))),
    "uniform": (em.StandardPrior(em.Uniform(-0.5, 3.0)), (up.UNIFORM, (-0.5, 3.0))),
    "beta": (em.StandardPrior(em.Beta(2.0, 3.0)), (up.BETA, (2.0, 3.0))),
    "cauchy": (em.StandardPrior(em.Cauchy(0.3, 1.5)), (up.CAUCHY, (0.3, 1.5))),
    "improper_pos": (em.ImproperPosPrior(), (up.IMPROPER_POS, ())),
    "product": (em.ProductPrior([em.Normal(0.5, 2.0), em.Gamma(2.0, 0.5)], [1, 1]),
                (up.PRODUCT_NORMAL_GAMMA, (0.5, 2.0, 2.0, 0.5))),
}


def _walk_update(walk, coords, prior, pos=None):
    n = len(coords)
    pos = [False] * (n - 1) + [True] if pos is None else pos
    if walk == "uniform":
        return em.RandomWalkUpdate(em.UniformRandomWalk([0.15] * n, pos), coords, prior=prior,
                                   adpt=em.AdaptationUnifRW([0.0] * n, adapt_every_k_steps=4, scale=0.02, offset=1.0))
    S = 0.01 * np.eye(n)
    if walk == "gauss":
        return em.RandomWalkUpdate(em.GaussianRandomWalk(S, pos), coords, prior=prior)
    return em.RandomWalkUpdate(em.GaussianRandomWalkMix(S, S, 0.3, pos), coords, prior=prior,
                               adpt=em.HaarioTypeAdaptation([0.0] * n, adapt_every_k_steps=3))


def _pair(name, walk, coords):
    builtin, (src, pp) = PRIORS[name]
    user = em.DevicePrior(src, params=pp, n_coords=len(coords))
    return [_walk_update(walk, coords, builtin)], [_walk_update(walk, coords, user)]


def _gsn1d(n=2000, seed=1):
    x = 0.45 + 0.5 * np.random.default_rng(seed).standard_normal(n)
    return x, np.array([0.45, 0.3])


@pytest.mark.parametrize("walk", ["uniform", "gauss", "mix"])
@pytest.mark.parametrize("name", sorted(PRIORS))
def test_restated_priors_give_the_builtin_bits_gsn1d(name, walk):
    x, t0 = _gsn1d()
    Cn, M = 96, 25
    a_ups, b_ups = _pair(name, walk, [1, 2])
    law = em.GsnTargetLaw([0.0])
    steps = list(em.MCMCSchedule(M, 1))
    a = _run(law, a_ups, x, t0, Cn, steps, 10)
    b = _run(law, b_ups, x, t0, Cn, steps, 10)
    _assert_same(a, b)
    assert 0.05 < a["accepted"].mean() < 0.95


@pytest.mark.parametrize("walk", ["gauss", "mix"])
@pytest.mark.parametrize("name", ["normal", "cauchy", "uniform"])
def test_restated_priors_give_the_builtin_bits_gsn_d2(name, walk):
    # GsnTargetLaw d = 2 (theta = [mu; vec Sigma], the general-d law): the walk with the prior moves mu, a
    # uniform walk moves the diagonal of Sigma, so the law constants of every proposal change
    rng = np.random.default_rng(7)
    L = np.linalg.cholesky(np.array([[1.0, 0.3], [0.3, 0.5]]))
    x = np.array([0.5, -0.2]) + rng.standard_normal((2000, 2)) @ L.T
    t0 = np.array([0.4, -0.1, 1.0, 0.3, 0.3, 0.5])
    builtin, (src, pp) = PRIORS[name]
    user = em.DevicePrior(src, params=pp, n_coords=2)
    diag = lambda: em.RandomWalkUpdate(em.UniformRandomWalk([0.05, 0.05], [True, True]), [3, 6],
                                       prior=em.ImproperPosPrior())
    law = em.GsnTargetLaw([0.0, 0.0])
    assert law.abi_law() == _abi.LAW_GSN_MV
    steps = list(em.MCMCSchedule(25, 2))
    a = _run(law, [_walk_update(walk, [1, 2], builtin, [False, False]), diag()], x, t0, 96, steps, 10)
    b = _run(law, [_walk_update(walk, [1, 2], user, [False, False]), diag()], x, t0, 96, steps, 10)
    _assert_same(a, b)
    assert 0.05 < a["accepted"].mean() < 0.95


def _logistic_data(n=600, d=4, seed=4):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, d)) / math.sqrt(d)
    beta = rng.standard_normal(d)
    y = (rng.random(n) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
    return X, y, beta


@pytest.mark.parametrize("walk", ["uniform", "gauss", "mix"])
@pytest.mark.parametrize("name", ["normal", "cauchy", "uniform"])
def test_restated_priors_give_the_builtin_bits_logistic(name, walk):
    X, y, beta = _logistic_data()
    Cn, M = 64, 20
    law = em.LogisticLaw(4)
    builtin, (src, pp) = PRIORS[name]
    mk = lambda pr, c: _walk_update(walk, c, pr)
    user = em.DevicePrior(src, params=pp, n_coords=2)
    steps = list(em.MCMCSchedule(M, 2))
    th0 = np.array([0.1, 0.2, 0.3, 0.4])
    a = _run(law, [mk(builtin, [1, 2]), mk(em.StandardPrior(em.Normal(0.0, 3.0)), [3, 4])], X, th0, Cn, steps, 8, y=y)
    b = _run(law, [mk(user, [1, 2]), mk(em.StandardPrior(em.Normal(0.0, 3.0)), [3, 4])], X, th0, Cn, steps, 8, y=y)
    _assert_same(a, b)


def test_restated_priors_give_the_builtin_bits_hier_and_device_law():
    # HierNormalLaw: walks on mu (Normal) and tau (ImproperPos) next to MALA on the group means
    G = 4
    rng = np.random.default_rng(5)
    yv = np.concatenate([rng.standard_normal(200) + g * 0.3 for g in range(G)])
    grp = np.repeat(np.arange(G), 200).astype(np.float64)
    th0 = np.concatenate([0.3 * np.arange(G), [0.2, 1.0]])
    law = em.HierNormalLaw(G)
    steps = list(em.MCMCSchedule(20, 3))

    def ups(mu_prior, tau_prior):
        return [em.MALAUpdate(0.05, list(range(1, G + 1))),
                em.RandomWalkUpdate(em.UniformRandomWalk([0.3]), [G + 1], prior=mu_prior),
                em.RandomWalkUpdate(em.UniformRandomWalk([0.3], [True]), [G + 2], prior=tau_prior)]
    a = _run(law, ups(em.StandardPrior(em.Normal(0.5, 2.0)), em.ImproperPosPrior()), yv, th0, 64, steps, 9, y=grp)
    b = _run(law, ups(em.DevicePrior(up.NORMAL, params=(0.5, 2.0)), em.DevicePrior(up.IMPROPER_POS)), yv, th0, 64,
             steps, 9, y=grp)
    _assert_same(a, b)
    # a DeviceLaw (the Gaussian law restated) under a Gaussian walk with a restated Gamma prior on both
    x, t0 = _gsn1d()
    dl = em.DeviceLaw(ul.GSN1D, 2, 1)
    a_ups, b_ups = _pair("gamma", "mix", [1, 2])
    s1 = list(em.MCMCSchedule(20, 1))
    _assert_same(_run(dl, a_ups, x[:, None], t0, 64, s1, 7), _run(dl, b_ups, x[:, None], t0, 64, s1, 7))


def test_uniform_prior_redraws_inside_the_prior_kernel():
    x, t0 = _gsn1d()
    Cn, M = 128, 30
    wide = lambda pr: [em.RandomWalkUpdate(em.UniformRandomWalk([1.5]), [1], prior=pr)]
    steps = list(em.MCMCSchedule(M, 1))
    a = _run(em.GsnTargetLaw([0.0]), wide(em.StandardPrior(em.Uniform(0.3, 0.6))), x, t0, Cn, steps, 30)
    b = _run(em.GsnTargetLaw([0.0]), wide(em.DevicePrior(up.UNIFORM, params=(0.3, 0.6))), x, t0, Cn, steps, 30)
    c = _run(em.GsnTargetLaw([0.0]), wide(em.ImproperPrior()), x, t0, Cn, steps, 30)
    _assert_same(a, b)
    mu_prop = b["theta_prop"][:, 0, :]
    assert np.all((mu_prop >= 0.3) & (mu_prop <= 0.6))           # every proposal was redrawn into [a, b]
    assert not np.array_equal(mu_prop, c["theta_prop"][:, 0, :])  # ... which the unconstrained walk is not


def test_replay_parity_with_the_builtin_prior_still_holds():
    x, t0 = _gsn1d()
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.1, 0.1], [False, True]), [1, 2],
                               prior=em.StandardPrior(em.Uniform(-0.5, 3.0)))]
    rep = replay_compare(x, 64, 20, seed=3, updates=ups, law=em.GsnTargetLaw([0.0]), theta_init=np.repeat(t0[:, None], 64, 1))
    assert rep["accept_mismatch"] == 0 and rep["theta_bitexact"], rep


@pytest.mark.parametrize("gradient", [True, "forward"])
def test_mala_restated_normal_gives_the_builtin_bits(gradient):
    # sigma = 2: a power of two, so that the forward-mode tangent (1/sd) z equals (th - m) / sd^2 exactly
    X, y, beta = _logistic_data(d=4)
    src = up.NORMAL if gradient is True else up.NORMAL_FORWARD
    mk = lambda pr: [em.MALAUpdate(0.2, [1, 2, 3, 4], prior=pr,
                                   adpt=em.AdaptationMALA(adapt_every_k_steps=5, scale=0.01, offset=1.0))]
    steps = list(em.MCMCSchedule(30, 1))
    th0 = np.zeros(4)
    a = _run(em.LogisticLaw(4), mk(em.StandardPrior(em.Normal(0.5, 2.0))), X, th0, 64, steps, 11, y=y)
    b = _run(em.LogisticLaw(4), mk(em.DevicePrior(src, gradient=gradient, params=(0.5, 2.0))), X, th0, 64, steps, 11, y=y)
    _assert_same(a, b)
    assert 0.1 < b["accepted"].mean() < 0.99


@pytest.mark.parametrize("src,gradient,pp", [(up.LAPLACE, True, (0.0, 0.5)), (up.STUDENT_T_FORWARD, "forward", (3.0, 1.0))])
def test_mala_laplace_and_student_t_on_logistic(src, gradient, pp):
    X, y, beta = _logistic_data(n=2000, d=4, seed=9)
    ups = [em.MALAUpdate(0.15, [1, 2, 3, 4], prior=em.DevicePrior(src, gradient=gradient, params=pp),
                         adpt=em.AdaptationMALA(adapt_every_k_steps=10, scale=0.01, offset=1.0))]
    out = _run(em.LogisticLaw(4), ups, X, np.zeros(4), 256, list(em.MCMCSchedule(300, 1)), 100, y=y)
    assert all(rc == 0 for rc in out["rc"])
    assert 0.3 < out["accepted"][100:].mean() < 0.99
    post = out["theta"][150:].mean(axis=(0, 2))
    assert np.all(np.isfinite(post)) and np.max(np.abs(post - beta)) < 1.0


def _laplace_ref(th, m, b):
    import mpmath as mp
    lp = mp.fsum(-abs(mp.mpf(t) - m) / b - mp.log(2 * mp.mpf(b)) for t in th)
    return lp, [-mp.sign(mp.mpf(t) - m) / b for t in th]


def _student_t_ref(th, nu, s):
    import mpmath as mp
    nu, s = mp.mpf(nu), mp.mpf(s)
    c = mp.loggamma((nu + 1) / 2) - mp.loggamma(nu / 2) - mp.log(nu * mp.pi) / 2 - mp.log(s)
    lp = mp.fsum(c - (nu + 1) / 2 * mp.log1p((mp.mpf(t) / s) ** 2 / nu) for t in th)
    return lp, [-(nu + 1) * mp.mpf(t) / (s * s * nu + mp.mpf(t) ** 2) for t in th]


@pytest.mark.parametrize("src,gradient,pp,ref", [(up.LAPLACE, True, (0.1, 0.5), _laplace_ref),
                                                  (up.STUDENT_T_FORWARD, "forward", (3.0, 1.5), _student_t_ref)])
def test_mala_prior_value_and_gradient_against_extended_precision(src, gradient, pp, ref):
    # lp and grad lp as the MALA kernels read them (extmcmc_eval_user_prior runs the same gradient kernel),
    # at the initial states and at the chains' states after MALA steps, against 50-digit arithmetic
    import mpmath as mp
    mp.mp.dps = 50
    X, y, _ = _logistic_data(n=2000, d=4, seed=9)
    Cn = 128
    th0 = np.random.default_rng(3).standard_normal((4, Cn))
    ups = [em.MALAUpdate(0.15, [1, 2, 3, 4], prior=em.DevicePrior(src, gradient=gradient, params=pp),
                         adpt=em.AdaptationMALA(adapt_every_k_steps=10, scale=0.01, offset=1.0))]
    g = _session(em.LogisticLaw(4), ups, X, th0, Cn, y=y, n_steps_hint=40)
    for rounds in range(2):
        th, _ = g.state()
        lp, gr = np.empty(Cn), np.empty((4, Cn))
        g.ck(g.lib.extmcmc_eval_user_prior(g.h, 0, _abi.dptr(lp), _abi.dptr(gr)))
        for c in range(Cn):
            rlp, rgr = ref(th[:, c], *pp)
            assert abs(lp[c] - float(rlp)) <= 1e-12 * max(1.0, abs(float(rlp))), (c, lp[c], rlp)
            for i in range(4):
                assert abs(gr[i, c] - float(rgr[i])) <= 1e-12 * max(1.0, abs(float(rgr[i]))), (c, i, gr[i, c], rgr[i])
        if rounds == 0:
            out = g.run(list(em.MCMCSchedule(40, 1)))
            assert out["rc"] == 0 and 0.2 < out["accepted"].mean() < 0.99
    g.close()


def test_laplace_posterior_mean_matches_quadrature():
    from scipy import integrate
    rng = np.random.default_rng(21)
    var, n = 1.0, 6
    x = 1.2 + rng.standard_normal(n)
    m, b = 0.0, 0.5
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.8]), [1], prior=em.DevicePrior(up.LAPLACE, params=(m, b)))]
    Cn, M = 4096, 400
    out = _run(em.GsnTargetLaw([0.0]), ups, x, np.array([0.0, var]), Cn, list(em.MCMCSchedule(M, 1)), 100)
    draws = out["theta"][200:, 0, :]            # [iterations][chains]
    chain_means = draws.mean(axis=0)
    est, mcse = chain_means.mean(), chain_means.std(ddof=1) / math.sqrt(Cn)
    logpost = lambda mu: -0.5 * np.sum((x - mu) ** 2) / var - abs(mu - m) / b
    lo, hi = -10.0, 10.0
    ref_max = max(logpost(t) for t in np.linspace(lo, hi, 2001))
    z = integrate.quad(lambda t: math.exp(logpost(t) - ref_max), lo, hi, points=[m], limit=200)[0]
    mean = integrate.quad(lambda t: t * math.exp(logpost(t) - ref_max), lo, hi, points=[m], limit=200)[0] / z
    assert abs(est - mean) < 3 * mcse, (est, mean, mcse)


def _plumbing_ups():
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.1]), [1], prior=em.DevicePrior(up.NORMAL, params=(0.5, 2.0))),
            em.RandomWalkUpdate(em.UniformRandomWalk([0.1], [True]), [2],
                                prior=em.DevicePrior(up.GAMMA, params=(2.0, 0.5)),
                                adpt=em.AdaptationUnifRW([0.0], adapt_every_k_steps=3, scale=0.02, offset=1.0))]


def test_graphs_block_lengths_and_chain_split_give_the_same_bits():
    x, t0 = _gsn1d()
    Cn, M = 80, 21
    law = em.GsnTargetLaw([0.0])
    steps = list(em.MCMCSchedule(M, 2))
    ref = _run(law, _plumbing_ups(), x, t0, Cn, steps, len(steps))
    for block in (1, 7, len(steps)):
        for graphs in (0, 1):
            _assert_same(ref, _run(law, _plumbing_ups(), x, t0, Cn, steps, block, use_graphs=graphs))
    half = Cn // 2
    parts = [_run(law, _plumbing_ups(), x, t0, half, steps, 7, chain_offset=o) for o in (0, half)]
    for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted"):
        assert np.array_equal(np.concatenate([p[k] for p in parts], axis=-1), ref[k]), k


def test_checkpoint_resume_in_a_fresh_handle():
    x, t0 = _gsn1d()
    Cn = 64
    law = em.GsnTargetLaw([0.0])
    steps = list(em.MCMCSchedule(20, 2))
    ref = _run(law, _plumbing_ups(), x, t0, Cn, steps, 20)
    g = _session(law, _plumbing_ups(), x, t0, Cn, n_steps_hint=20)
    first = g.run(steps[:20])
    n = C.c_int64()
    g.ck(g.lib.extmcmc_checkpoint_size(g.h, C.byref(n)))
    blob = (C.c_uint8 * n.value)()
    g.ck(g.lib.extmcmc_checkpoint_save(g.h, blob, n.value))
    g.close()
    h = _session(law, _plumbing_ups(), x, t0, Cn, n_steps_hint=20)
    h.ck(h.lib.extmcmc_checkpoint_load(h.h, blob, n.value))
    h.seq = 20
    second = h.run(steps[20:])
    h.close()
    for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted"):
        assert np.array_equal(np.concatenate([first[k], second[k]]), ref[k]), k


def test_launch_counts():
    x, t0 = _gsn1d()
    law = em.GsnTargetLaw([0.0])
    M = 12
    steps = list(em.MCMCSchedule(M, 1))
    rw = lambda pr: [em.RandomWalkUpdate(em.UniformRandomWalk([0.1]), [1], prior=pr)]
    a = _run(law, rw(em.StandardPrior(em.Normal(0.5, 2.0))), x, t0, 64, steps, M)
    b = _run(law, rw(em.DevicePrior(up.NORMAL, params=(0.5, 2.0))), x, t0, 64, steps, M)
    # one prior kernel per element, and the proposals no longer ride on the previous accept kernel
    assert b["launches"] - a["launches"] == M + (M - 1)
    X, y, _ = _logistic_data()
    mala = lambda pr: [em.MALAUpdate(0.1, [1, 2, 3, 4], prior=pr)]
    c = _run(em.LogisticLaw(4), mala(em.StandardPrior(em.Normal(0.5, 2.0))), X, np.zeros(4), 64, steps, M, y=y)
    d = _run(em.LogisticLaw(4), mala(em.DevicePrior(up.NORMAL, gradient=True, params=(0.5, 2.0))), X, np.zeros(4),
             64, steps, M, y=y)
    assert d["launches"] - c["launches"] == 2 * M


def test_refusals():
    x, t0 = _gsn1d()
    law = em.GsnTargetLaw([0.0])
    steps = list(em.MCMCSchedule(2, 1))
    # no prior installed
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.1]), [1], prior=em.DevicePrior(up.NORMAL, params=(0.5, 2.0)))]
    g = GpuSession(law, ups, x, t0, 64)
    with pytest.raises(_abi.ExtMCMCError) as e:
        g.run(steps)
    assert e.value.code == _abi.EINVAL
    g.close()
    # a prior without gradient under MALA
    X, y, _ = _logistic_data()
    ups = [em.MALAUpdate(0.1, [1, 2], prior=em.DevicePrior(up.UNIFORM, params=(-5.0, 5.0), n_coords=2))]
    g = GpuSession(em.LogisticLaw(4), ups, X, np.zeros(4), 64, y=y)
    assert ups[0].prior.abi_attach(g.lib, g.h, 0) == _abi.EUNSUPPORTED
    g.close()
    # the persistent block kernels
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.1]), [1], prior=em.DevicePrior(up.NORMAL, params=(0.5, 2.0)))]
    g = _session(law, ups, x, t0, 64, sweep_variant=3)
    with pytest.raises(_abi.ExtMCMCError) as e:
        g.run(steps)
    assert e.value.code == _abi.EUNSUPPORTED
    g.close()
    # observation sharding over several ranks
    with pytest.raises(_abi.ExtMCMCError) as e:
        GpuSession(law, ups, x, t0, 64, shard_mode=_abi.SHARD_OBS, world_size=2)
    assert e.value.code == _abi.EUNSUPPORTED and "user priors" in str(e.value)
    # the value and gradient of a prior without gradient cannot be evaluated
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.1]), [1], prior=em.DevicePrior(up.NORMAL, params=(0.5, 2.0)))]
    g = _session(law, ups, x, t0, 64)
    lp, gr = np.empty(64), np.empty(64)
    assert g.lib.extmcmc_eval_user_prior(g.h, 0, _abi.dptr(lp), _abi.dptr(gr)) == _abi.EUNSUPPORTED
    g.close()
