"""Forward-mode gradients of user-defined laws (DeviceLaw(..., gradient="forward"),
EXTMCMC_USER_GRAD_FORWARD) on the B200: every forward kernel against the extended-precision gradients
of tests/user_laws.py, the log-likelihood of a gradient sweep bit-identical to the value sweep's, the
forward against the hand-written gradient, MALA decisions under replayed randomness, a conjugate
posterior of a law that has no hand-written gradient, bit-identical launch variants and checkpoint /
resume."""
import ctypes as C
import math

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws_forward as uf
from tests.parity import GpuSession, compare_histories
from tests.test_gpu_user_law import _data, _theta

pytestmark = pytest.mark.gpu

G_TOL = 1e-12          # |grad - ref| <= G_TOL * sum_j |g_j|, per chain and coordinate
HAND_TOL = 1e-13       # forward against hand-written, same normalisation
NT = 128
ALL_FORWARD = {"chains_r1_f", "chains_r2_f", "chains_r4_f", "lanes_f"}
_launched = set()
_cases_done = []


def _session(src, P, D, updates, X, th0, Cn, seed=0, gradient="forward", **cfg):
    """GpuSession of a DeviceLaw, installed the way the Python mirror installs it."""
    law = em.DeviceLaw(src, P, D, gradient=gradient)
    g = GpuSession(law, updates, X, th0, Cn, seed=seed, **cfg)
    g.ck(law.abi_attach(g.lib, g.h))
    return g


def _ups():
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.01]), [1])]


def _law_data(law, N, D, seed):
    if law == "poisson_rate":
        return np.random.default_rng(seed).poisson(4.0, (N, 1)).astype(np.float64)
    return _data(law, N, D, seed=seed)


def _law_theta(law, P, Cn, seed):
    if law == "poisson_rate":
        return 4.0 * np.exp(0.2 * np.random.default_rng(seed).standard_normal((1, Cn)))
    return _theta(law, P, Cn, seed=seed)


def _reference(law, th, X, chunk=32):
    """ll [C], grad [P, C] and sum_j |g_j| [P, C] in np.longdouble, as float64."""
    terms = uf.LAWS[law][3]
    Cn = th.shape[1]
    ll, gr, gra = np.empty(Cn), np.empty((th.shape[0], Cn)), np.empty((th.shape[0], Cn))
    for lo in range(0, Cn, chunk):
        t, g = terms(th[:, lo:lo + chunk], X, dtype=np.longdouble)
        ll[lo:lo + chunk] = t.sum(axis=0)
        gr[:, lo:lo + chunk] = g.sum(axis=1)
        gra[:, lo:lo + chunk] = np.abs(g).sum(axis=1)
    return ll, gr, gra


def _kernel(variant):
    return "lanes_f" if variant == "user_lanes" else "chains_r" + variant[len("user_chains_R"):] + "_f"


# (law, D): P = 1, 2, 2, 3, 8; D = 3 is an odd obs_dim (a tile is not a power of two of rows)
LAW_SHAPES = [("poisson_rate", 1), ("gsn1d", 1), ("logistic", 3), ("poisson_reg", 3), ("poisson_reg", 8)]
# forced chains R = 1 / 2 / 4 and lanes; C = 701 leaves the last CTA ragged under every mapping
VARIANTS = [11, 12, 14, 2]
N_ROWS = 3001


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("law,D", LAW_SHAPES)
def test_forward_gradient_every_kernel_every_chain(law, D, variant):
    src, hand, Pf, _ = uf.LAWS[law]
    P = Pf(D)
    Cn = 701
    X = _law_data(law, N_ROWS, D, seed=21)
    th = _law_theta(law, P, Cn, seed=22)
    g = _session(src, P, D, _ups(), X, th, Cn, sweep_variant=variant)
    v = g.variant()
    rmax = 4 if 4 * (P + 1) ** 2 <= 40 else 2 if 2 * (P + 1) ** 2 <= 40 else 1
    assert v == ("user_lanes" if variant == 2 else f"user_chains_R{min(variant - 10, rmax)}"), v
    ll_v = g.eval_loglik()
    ll_g, gr = g.eval_grad()
    assert g.lib.extmcmc_sync(g.h) == _abi.OK
    _launched.add(_kernel(v))
    # the value parts of the dual operations are the value sweep's: the same bits, every chain
    assert np.array_equal(ll_g, ll_v), np.abs(ll_g - ll_v).max()
    llw, grw, gra = _reference(law, th, X)
    e_g = np.abs(gr - grw) / (G_TOL * np.maximum(gra, 1e-300))
    e_ll = np.abs(ll_v - llw) / (G_TOL * np.abs(llw).clip(1.0))
    print(f"{law} P={P} D={D} {v}: grad err / tol {e_g.max():.3g}, ll err / tol {e_ll.max():.3g}")
    assert e_g.max() <= 1, (np.unravel_index(np.argmax(e_g), e_g.shape), e_g.max())
    g.close()
    if hand is not None:
        # the same law with its hand-written gradient, same kernel mapping
        h = GpuSession(em.DeviceLaw(hand, P, D, gradient=True), _ups(), X, th, Cn, sweep_variant=variant)
        h.ck(h.lib.extmcmc_set_user_law(h.h, hand.encode(), _abi.USER_GRAD_HAND))
        ll_h, gr_h = h.eval_grad()
        assert h.lib.extmcmc_sync(h.h) == _abi.OK
        e_h = np.abs(gr - gr_h) / (HAND_TOL * np.maximum(gra, 1e-300))
        print(f"  against the hand-written gradient: err / tol {e_h.max():.3g}")
        assert e_h.max() <= 1, e_h.max()
        h.close()
    _cases_done.append((law, variant))


def test_every_forward_kernel_was_launched():
    if len(_cases_done) < len(LAW_SHAPES) * len(VARIANTS):
        pytest.skip("needs every case of test_forward_gradient_every_kernel_every_chain in the same run")
    assert _launched == ALL_FORWARD, ALL_FORWARD - _launched


def test_forward_gradient_many_segments_planner_choice():
    # 2^20 + 3 rows over many segments and tiles, the planner's own mapping at 4096 and at 5 chains
    law, D = "poisson_reg", 5
    P = D
    X = _data(law, 2**20 + 3, D, seed=5)
    for Cn in (4096, 5):
        th = _theta(law, P, Cn, seed=6)
        g = _session(uf.POISSON_REG, P, D, _ups(), X, th, Cn)
        ll_g, gr = g.eval_grad()
        assert np.array_equal(ll_g, g.eval_loglik())
        sub = np.unique(np.linspace(0, Cn - 1, min(Cn, 8)).astype(int))
        _, grw, gra = _reference(law, th[:, sub], X)
        e = np.abs(gr[:, sub] - grw) / (G_TOL * gra)
        print(f"{g.variant()} C={Cn}: grad err / tol {e.max():.3g}")
        assert e.max() <= 1, e.max()
        g.close()


# ---- MALA ----------------------------------------------------------------------------------------------

def _poisson_reg_grad(th, X):
    """d ll / d theta [P, C] in fp64 (numpy), the MALA correction's gradient for the near-tie margin."""
    P = th.shape[0]
    e = th[0][None, :] + X[:, :P - 1] @ th[1:]
    r = X[:, P - 1:P] - np.exp(e)
    return np.concatenate([r.sum(axis=0)[None], X[:, :P - 1].T @ r], axis=0)


def test_mala_forward_against_hand_gradient_under_replay():
    D = P = 3
    Cn, M, tau = 256, 200, 0.02
    X = _data("poisson_reg", 2000, D, seed=8)
    th0 = 0.3 * np.random.default_rng(9).standard_normal((P, Cn))
    ups = [em.MALAUpdate(tau, [1, 2, 3])]
    steps = list(em.MCMCSchedule(M, 1))
    # the randomness to replay: the proposals of a run under the hand gradient's own Philox stream and
    # independent Exp(1) draws
    src = GpuSession(em.DeviceLaw(uf.LAWS["poisson_reg"][1], P, D, gradient=True), ups, X, th0, Cn, seed=4,
                     n_steps_hint=M)
    src.ck(src.lib.extmcmc_set_user_law(src.h, uf.LAWS["poisson_reg"][1].encode(), _abi.USER_GRAD_HAND))
    props = np.ascontiguousarray(src.run(steps)["theta_prop"])
    src.close()
    exps = np.random.default_rng(10).exponential(size=(M, Cn))
    runs = {}
    for mode in ("hand", "forward"):
        s = uf.LAWS["poisson_reg"][1] if mode == "hand" else uf.POISSON_REG
        g = _session(s, P, D, ups, X, th0, Cn, seed=4, gradient=True if mode == "hand" else "forward",
                     n_steps_hint=M)
        runs[mode] = g.run(steps, replay=(props, exps))
        runs[mode]["variant"] = g.variant()
        g.close()
    h, f = runs["hand"], runs["forward"]
    # the hand run in the role of the reference: its log acceptance ratios for the near-tie margin
    prev = np.concatenate([th0[None], h["theta"][:-1]])
    ll_prev = np.concatenate([np.full((1, Cn), -np.inf), h["ll"][:-1]])
    llr = np.empty((M, Cn))
    for s in range(M):
        ga, gb = _poisson_reg_grad(prev[s], X), _poisson_reg_grad(h["theta_prop"][s], X)
        a, b = prev[s], h["theta_prop"][s]
        qf = -((b - a - tau * tau / 2 * ga) ** 2).sum(axis=0) / (2 * tau * tau)
        qb = -((a - b - tau * tau / 2 * gb) ** 2).sum(axis=0) / (2 * tau * tau)
        llr[s] = h["ll_prop"][s] - ll_prev[s] + qb - qf
    rep = compare_histories(dict(h, exp_draws=exps, llr=llr), f)
    print(rep, h["variant"], "accept rate", h["accepted"].mean())
    assert 0.2 < h["accepted"][1:].mean() < 0.95
    assert rep["accept_mismatch"] == 0 and rep["theta_bitexact"] and rep["ll_rel_err"] < 1e-12, rep


def test_mala_posterior_of_a_law_without_hand_gradient():
    # POISSON_RATE has no logpdf_grad; flat prior on the rate: the posterior is Gamma(1 + sum y, N)
    rng = np.random.default_rng(3)
    N = 200
    y = rng.poisson(4.0, N).astype(np.float64)
    law = em.DeviceLaw(uf.POISSON_RATE, 1, 1, gradient="forward")
    up = [em.MALAUpdate(0.12, [1])]
    Cn, M, burn = 256, 4000, 500
    mcmc = em.MCMC(up, backend=em.CUDAMCMCBackend(n_chains=Cn, seed=3, block_len=200))
    ws, _ = em.run_(mcmc, M, dict(P=law, obs=y[:, None]), [4.0])
    tr = ws.sub_ws.state_history[burn:, 0, 0]            # [M - burn, C]
    shape, rate = 1.0 + y.sum(), float(N)
    mean_w, var_w = shape / rate, shape / rate ** 2
    ess = em.ess_geyer(tr).sum()
    mcse_mean = math.sqrt(tr.var() / ess)
    mcse_var = math.sqrt(((tr - tr.mean()) ** 2).var() / ess)
    print(f"mean {tr.mean():.6g} (want {mean_w:.6g}, mcse {mcse_mean:.3g}), var {tr.var():.6g} "
          f"(want {var_w:.6g}, mcse {mcse_var:.3g}), ess {ess:.0f}")
    assert abs(tr.mean() - mean_w) < 3 * mcse_mean, (tr.mean(), mean_w, mcse_mean)
    assert abs(tr.var() - var_w) < 3 * mcse_var, (tr.var(), var_w, mcse_var)
    ws.close()


# ---- determinism -------------------------------------------------------------------------------------------

def _det_problem():
    D = P = 4
    X = _data("poisson_reg", 5000, D, seed=4)
    th0 = 0.01 * np.random.default_rng(2).standard_normal((P, 300))
    ups = [em.RandomWalkUpdate(em.UniformRandomWalk([0.02, 0.02]), [1, 2]),
           em.MALAUpdate(0.05, [2, 3, 4], prior=em.StandardPrior(em.Normal(0.0, 10.0)),
                         adpt=em.AdaptationMALA(adapt_every_k_steps=5, scale=0.01, offset=1.0))]
    return D, P, X, th0, ups


def test_launch_variants_are_bit_identical():
    D, P, X, th0, ups = _det_problem()
    steps = list(em.MCMCSchedule(12, 2))
    out = {}
    for name, cfg, block, splits in [("eager_all", dict(use_graphs=0), 24, [(0, 300)]),
                                     ("graph_all", dict(use_graphs=1), 24, [(0, 300)]),
                                     ("graph_b4", dict(use_graphs=1), 4, [(0, 300)]),
                                     ("eager_b1", dict(use_graphs=0), 1, [(0, 300)]),
                                     ("split", dict(use_graphs=1), 24, [(0, 130), (130, 300)])]:
        th, ll = [], []
        for lo, hi in splits:
            g = _session(uf.POISSON_REG, P, D, ups, X, np.ascontiguousarray(th0[:, lo:hi]), hi - lo, seed=7,
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


def test_checkpoint_resume():
    D, P, X, th0, ups = _det_problem()
    Cn, M = 300, 20
    s1 = list(em.MCMCSchedule(M, 2))
    a = _session(uf.POISSON_REG, P, D, ups, X, th0, Cn, seed=5, n_steps_hint=2 * M)
    a.run(s1[:M]); a.run(s1[M:])
    th_a, ll_a = a.state()
    b = _session(uf.POISSON_REG, P, D, ups, X, th0, Cn, seed=5, n_steps_hint=2 * M)
    b.run(s1[:M])
    n = C.c_int64()
    b.ck(b.lib.extmcmc_checkpoint_size(b.h, C.byref(n)))
    blob = (C.c_uint8 * n.value)()
    b.ck(b.lib.extmcmc_checkpoint_save(b.h, blob, n.value))
    c = _session(uf.POISSON_REG, P, D, ups, X, th0 * 0 + th0[:, :1], Cn, seed=5, n_steps_hint=2 * M)
    c.ck(c.lib.extmcmc_checkpoint_load(c.h, blob, n.value))
    c.seq = M
    c.run(s1[M:])
    th_c, ll_c = c.state()
    assert np.array_equal(th_a, th_c) and np.array_equal(ll_a, ll_c)
    # the same source under the hand-written contract is another law: its blob is refused
    d = GpuSession(em.DeviceLaw(uf.LAWS["poisson_reg"][1], P, D, gradient=True), ups, X, th0, Cn, seed=5,
                   n_steps_hint=2 * M)
    d.ck(d.lib.extmcmc_set_user_law(d.h, uf.LAWS["poisson_reg"][1].encode(), _abi.USER_GRAD_HAND))
    assert d.lib.extmcmc_checkpoint_load(d.h, blob, n.value) == _abi.EINVAL
    for s in (a, b, c, d):
        s.close()


def test_forward_mode_limit_on_a_handle():
    law = em.DeviceLaw(uf.POISSON_REG, 2, 2, gradient="forward")
    X = _data("poisson_reg", 100, 2, seed=1)
    g = GpuSession(law, _ups(), X, np.zeros(2), 8)
    # the handle is for P = 2: forward mode is fine there; eval_grad works without a hand gradient
    g.ck(law.abi_attach(g.lib, g.h))
    ll, gr = g.eval_grad()
    assert np.isfinite(gr).all()
    g.close()
    X17 = _data("poisson_reg", 100, 17, seed=1)
    hand = em.DeviceLaw(uf.LAWS["poisson_reg"][1], 17, 17, gradient=True)
    g = GpuSession(hand, _ups(), X17, np.zeros(17), 8)
    assert g.lib.extmcmc_set_user_law(g.h, uf.POISSON_REG.encode(), _abi.USER_GRAD_FORWARD) == _abi.EUNSUPPORTED
    assert b"n_params <= 16" in g.lib.extmcmc_last_error(g.h)
    g.close()
