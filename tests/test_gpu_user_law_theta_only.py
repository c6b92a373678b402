"""User-defined laws with parameter-only coordinates on the B200 (DeviceLaw(..., theta_only=...),
extmcmc_set_user_law_theta_only): every kernel the planner can pick against the extended-precision
references and against the undeclared law, the row-sum cache on against off (EXTMCMC_DATA_CACHE) bit for
bit under the library's own Philox stream, the sweeps it saves, replay parity of the declared hierarchical
restatement against the oracle's built-in law, checkpoint / resume, and a row-free proposal outside the
law's domain."""
import ctypes as C

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from oracle import oracle as orc
from tests import user_laws_theta as ut
from tests.parity import GpuSession, compare_histories
from tests.test_gpu_mala import _hier_theta0, _hier_updates

pytestmark = pytest.mark.gpu
G = ut.G
P = G + 2
TOL = 1e-12
ONLY = {"hier": (P - 1, P), "ridge": (P,)}   # mu, tau; log lambda


def _law(name, gradient, chunk=None, declared=True):
    hand, fwd, Df, _, _ = ut.LAWS[name]
    src = fwd if gradient == "forward" else hand
    return em.DeviceLaw(src, P, Df(P), gradient=gradient, chunk=chunk, theta_term=True,
                        theta_only=ONLY[name] if declared else None)


def _session(law, updates, X, th0, Cn, seed=0, **cfg):
    g = GpuSession(law, updates, X, th0, Cn, seed=seed, **cfg)
    g.ck(law.abi_attach(g.lib, g.h))
    return g


def _ups():
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.01]), [1])]


# ---- every kernel against extended precision and against the undeclared law ------------------------------

CASES = [("hier", False, None), ("hier", True, None), ("hier", "forward", None), ("hier", "forward", 3),
         ("hier", "forward", 5), ("ridge", True, None), ("ridge", "forward", None), ("ridge", "forward", 3)]


@pytest.mark.parametrize("variant", [11, 12, 14, 2])
@pytest.mark.parametrize("name,gradient,chunk", CASES)
def test_every_kernel_against_extended_precision(name, gradient, chunk, variant):
    for N in (3001, 7):
        X = ut.data(name, N, P, seed=21)
        Cn = 701
        th = ut.theta(name, P, Cn, seed=22)
        out = {}
        for declared in (True, False):
            g = _session(_law(name, gradient, chunk, declared), _ups(), X, th, Cn, sweep_variant=variant)
            v = g.variant()
            assert v == "user_lanes" if variant == 2 else v.startswith("user_chains_R"), v
            out[declared] = (g.eval_loglik(),) + (g.eval_grad() if gradient else ())
            assert g.lib.extmcmc_sync(g.h) == _abi.OK
            g.close()
        llw, lla, grw, gra = ut.reference(name, th, X)
        ll_v = out[True][0]
        assert (np.abs(ll_v - llw) / (TOL * lla)).max() <= 1, (N, v)
        assert (np.abs(ll_v - out[False][0]) / np.abs(out[False][0])).max() <= TOL, (N, v)
        if gradient:
            ll_g, gr = out[True][1:]
            if gradient == "forward":
                assert np.array_equal(ll_g, ll_v)
            assert (np.abs(ll_g - llw) / (TOL * lla)).max() <= 1, (N, v)
            assert (np.abs(gr - grw) / (TOL * np.maximum(gra, 1e-300))).max() <= 1, (N, v)
            gu = out[False][2]
            assert (np.abs(gr - gu) / (TOL * np.maximum(gra, 1e-300))).max() <= 1, (N, v)


# ---- the cache on against off ------------------------------------------------------------------------------

def _run(monkeypatch, cache, law, ups, X, th0, Cn, steps, block, seed=3, **cfg):
    monkeypatch.setenv("EXTMCMC_DATA_CACHE", "1" if cache else "0")
    g = _session(law, ups, X, th0, Cn, seed=seed, n_steps_hint=len(steps), **cfg)
    parts = [g.run(steps[b:b + block]) for b in range(0, len(steps), block)]
    out = {k: np.concatenate([q[k] for q in parts]) for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted")}
    out["rc"] = [q["rc"] for q in parts]
    out["eps"] = [g.eps(u) for u in range(1, len(ups) + 1)]
    out["stats"] = g.stats()
    out["state"] = g.state()
    g.close()
    return out


def _assert_same(a, b):
    for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert a["rc"] == b["rc"]
    assert all(np.array_equal(x, y) for x, y in zip(a["eps"], b["eps"]))
    for k, v in a["stats"].items():
        assert np.array_equal(v, b["stats"][k], equal_nan=True), k
    assert np.array_equal(a["state"][0], b["state"][0]) and np.array_equal(a["state"][1], b["state"][1])


def _ridge_updates(mala):
    beta = list(range(1, P))
    first = (em.MALAUpdate(0.02, beta, adpt=em.AdaptationMALA(adapt_every_k_steps=6, scale=0.004, offset=1.0)) if mala
             else em.RandomWalkUpdate(em.UniformRandomWalk([0.05] * len(beta)), beta))
    return [first, em.RandomWalkUpdate(em.UniformRandomWalk([0.3]), [P],
                                       adpt=em.AdaptationUnifRW([0.0], adapt_every_k_steps=5, scale=0.02, offset=1.0))]


HIER_LAWS = [(True, None), ("forward", None), ("forward", 3), ("forward", 5)]


@pytest.mark.parametrize("gradient,chunk", HIER_LAWS)
@pytest.mark.parametrize("extra_walk", [False, True])
def test_cache_on_and_off_give_the_same_bits_hier(monkeypatch, gradient, chunk, extra_walk):
    X, _ = ut.hier_data(400, seed=9, ragged=True)
    Cn, M = 300, 14
    ups = _hier_updates(G)
    if extra_walk:   # a walk on theta_1: moves a row coordinate, its accepted R is committed
        ups = ups + [em.RandomWalkUpdate(em.UniformRandomWalk([0.2]), [1])]
    th0 = _hier_theta0(G, Cn)
    steps = list(em.MCMCSchedule(M, len(ups), [(2, range(4, 7))]))
    law = _law("hier", gradient, chunk)
    for cfg, block in [(dict(use_graphs=0), 1), (dict(use_graphs=1), 4), (dict(use_graphs=1), 7),
                       (dict(use_graphs=0), len(steps))]:
        on = _run(monkeypatch, True, law, ups, X, th0, Cn, steps, block, **cfg)
        off = _run(monkeypatch, False, law, ups, X, th0, Cn, steps, block, **cfg)
        _assert_same(on, off)
        assert 0.05 < on["accepted"].mean() < 0.95
        assert np.isfinite(on["ll"][1:]).all()


@pytest.mark.parametrize("gradient", [True, "forward"])
@pytest.mark.parametrize("mala", [False, True])
def test_cache_on_and_off_give_the_same_bits_ridge(monkeypatch, gradient, mala):
    X = ut.data("ridge", 2000, P, seed=11)
    Cn, M = 256, 16
    ups = _ridge_updates(mala)
    th0 = ut.theta("ridge", P, Cn, seed=12)
    steps = list(em.MCMCSchedule(M, len(ups), [(1, range(5, 8))]))
    law = _law("ridge", gradient)
    for cfg, block in [(dict(use_graphs=1), 1), (dict(use_graphs=0), 4), (dict(use_graphs=1), len(steps))]:
        on = _run(monkeypatch, True, law, ups, X, th0, Cn, steps, block, **cfg)
        off = _run(monkeypatch, False, law, ups, X, th0, Cn, steps, block, **cfg)
        _assert_same(on, off)
        assert 0 < on["accepted"].mean() < 1


# ---- sweeps per iteration ----------------------------------------------------------------------------------

def _sweeps(monkeypatch, cache, law, ups, X, th0, Cn, M):
    monkeypatch.setenv("EXTMCMC_DATA_CACHE", "1" if cache else "0")
    steps = list(em.MCMCSchedule(M, len(ups)))
    g = _session(law, ups, X, th0, Cn, seed=5, n_steps_hint=len(steps), instrument=1)
    g.run(steps)
    ms, n = C.c_float(), C.c_int64()
    g.ck(g.lib.extmcmc_get_sweep_time(g.h, C.byref(ms), C.byref(n)))
    g.close()
    return n.value


@pytest.mark.parametrize("gradient", [True, "forward"])
def test_sweep_counts(monkeypatch, gradient):
    M = 10
    X, _ = ut.hier_data(300, seed=2)
    Cn = 256
    law = _law("hier", gradient)
    # cfg 4's schedule: MALA on theta_1..8, walks on mu and tau
    assert _sweeps(monkeypatch, True, law, _hier_updates(G), X, _hier_theta0(G, Cn), Cn, M) == M + 1
    assert _sweeps(monkeypatch, False, law, _hier_updates(G), X, _hier_theta0(G, Cn), Cn, M) == 4 * M
    Xr = ut.data("ridge", 1000, P, seed=3)
    thr = ut.theta("ridge", P, Cn, seed=4)
    law = _law("ridge", gradient)
    assert _sweeps(monkeypatch, True, law, _ridge_updates(False), Xr, thr, Cn, M) == M + 1
    assert _sweeps(monkeypatch, False, law, _ridge_updates(False), Xr, thr, Cn, M) == 2 * M


# ---- replay parity against the oracle's built-in law ---------------------------------------------------------

@pytest.mark.parametrize("gradient", [True, "forward"])
@pytest.mark.parametrize("Cn,ragged", [(200, False), (7, True)])
def test_replay_parity_declared_hier_cfg4(gradient, Cn, ragged):
    X, grp = ut.hier_data(256, seed=5, ragged=ragged)
    ups = _hier_updates(G)
    th0 = _hier_theta0(G, Cn)
    steps = list(em.MCMCSchedule(30, len(ups)))
    o = orc.Oracle(em.HierNormalLaw(G), ups, X[:, 0].copy(), th0, Cn, seed=12, y=grp)
    ro = o.run(steps, n_threads=8)
    g = _session(_law("hier", gradient), ups, X, th0, Cn, seed=12, n_steps_hint=len(steps), history_window=40)
    parts = [g.run(steps[b:b + 13], replay=(ro["proposals"][b:b + 13], ro["exp_draws"][b:b + 13]))
             for b in range(0, len(steps), 13)]
    rg = {k: np.concatenate([q[k] for q in parts]) for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted")}
    rep = compare_histories(ro, rg)
    if rep["chains_diverged"] == 0:
        so, sg = o.stats(), g.stats()
        rep["eps_bitexact"] = all(np.array_equal(o.eps(u), g.eps(u)) for u in range(1, len(ups) + 1))
        rep["moments_bitexact"] = bool(np.array_equal(so["mean"], sg["mean"]) and np.array_equal(so["cov"], sg["cov"]))
        rep["counts_equal"] = bool(np.array_equal(so["n_accept"], sg["n_accept"]))
    g.close()
    print(rep)
    assert rep["accept_mismatch"] == 0 and rep["theta_bitexact"] and rep["ll_rel_err"] < 1e-12, rep
    assert 0.02 < rep["accept_rate"] < 0.98, rep
    if rep["chains_diverged"] == 0:
        assert rep["eps_bitexact"] and rep["moments_bitexact"] and rep["counts_equal"], rep


# ---- checkpoint / resume -------------------------------------------------------------------------------------

def _save(g):
    n = C.c_int64()
    g.ck(g.lib.extmcmc_checkpoint_size(g.h, C.byref(n)))
    blob = (C.c_uint8 * n.value)()
    g.ck(g.lib.extmcmc_checkpoint_save(g.h, blob, n.value))
    return blob, n.value


@pytest.mark.parametrize("gradient", [True, "forward"])
def test_checkpoint_resume_and_other_declarations_are_refused(gradient):
    X, _ = ut.hier_data(200, seed=4)
    Cn, M = 150, 20
    ups = _hier_updates(G)
    th0 = _hier_theta0(G, Cn)
    s1 = list(em.MCMCSchedule(M, len(ups)))
    mk = lambda law, th: _session(law, ups, X, th, Cn, seed=5, n_steps_hint=2 * M, use_graphs=1)  # noqa: E731
    law = _law("hier", gradient)
    a = mk(law, th0)
    a.run(s1[:M])
    ra = a.run(s1[M:])
    th_a, ll_a = a.state()
    b = mk(law, th0)
    b.run(s1[:M])
    blob, n = _save(b)
    c = mk(law, th0 * 0 + th0[:, :1])
    c.ck(c.lib.extmcmc_checkpoint_load(c.h, blob, n))
    c.seq = M
    rc = c.run(s1[M:])
    th_c, ll_c = c.state()
    for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted"):
        assert np.array_equal(ra[k], rc[k]), k
    assert np.array_equal(th_a, th_c) and np.array_equal(ll_a, ll_c)
    # another declaration, and no declaration, are other programs: refused both ways
    hand, fwd, _, _, _ = ut.LAWS["hier"]
    src = fwd if gradient == "forward" else hand
    others = [em.DeviceLaw(src, P, 2, gradient=gradient, theta_term=True, theta_only=[P]),
              em.DeviceLaw(src, P, 2, gradient=gradient, theta_term=True)]
    for other in others:
        d = mk(other, th0)
        assert d.lib.extmcmc_checkpoint_load(d.h, blob, n) == _abi.EINVAL
        assert b"another user law" in d.lib.extmcmc_last_error(d.h)
        d.run(s1[:2])
        blob_d, n_d = _save(d)
        assert c.lib.extmcmc_checkpoint_load(c.h, blob_d, n_d) == _abi.EINVAL
        d.close()
    for s in (a, b, c):
        s.close()


# ---- a row-free proposal outside the domain ---------------------------------------------------------------

@pytest.mark.parametrize("gradient", [True, "forward"])
def test_row_free_proposal_outside_the_domain(monkeypatch, gradient):
    X, _ = ut.hier_data(300, seed=6)
    Cn = 96
    ups = _hier_updates(G)
    th0 = _hier_theta0(G, Cn)
    steps = list(em.MCMCSchedule(2, len(ups)))   # MALA, mu, tau; twice
    rng = np.random.default_rng(7)
    props = np.zeros((len(steps), G, Cn))
    for s, st in enumerate(steps):
        if st.pidx == 1:
            props[s, :G] = th0[:G] + 0.01 * rng.standard_normal((G, Cn))
        elif st.pidx == 2:
            props[s, 0] = th0[G] + 0.01 * rng.standard_normal(Cn)
        else:
            tau = th0[G + 1].copy()
            tau[::3] = -0.5          # tau <= 0: set_parameters is false
            props[s, 0] = tau
    exps = rng.exponential(size=(len(steps), Cn))
    out = {}
    for cache in (True, False):
        monkeypatch.setenv("EXTMCMC_DATA_CACHE", "1" if cache else "0")
        g = _session(_law("hier", gradient), ups, X, th0, Cn, seed=1, n_steps_hint=len(steps))
        r = g.run(steps, replay=(props, exps))
        out[cache] = (r, g.state())
        g.close()
    (r1, s1), (r0, s0) = out[True], out[False]
    assert r1["rc"] == r0["rc"] == _abi.EDOMAIN
    tau_steps = [s for s, st in enumerate(steps) if st.pidx == 3]
    for s in tau_steps:
        assert not r1["accepted"][s, ::3].any()
        assert np.isnan(r1["ll_prop"][s, ::3]).all()
    for k in ("theta", "theta_prop", "ll", "ll_prop", "accepted"):
        assert np.array_equal(r1[k], r0[k], equal_nan=True), k
    assert np.array_equal(s1[0], s0[0]) and np.array_equal(s1[1], s0[1])
