"""User-defined laws with a term of theta only on the B200 (DeviceLaw(..., theta_term=True),
extmcmc_set_user_law_ex): every kernel the planner can pick against the extended-precision references of
tests/user_laws_theta.py, the hierarchical restatement replayed against the oracle's built-in
hierarchical law under the cfg 4 schedule and run beside the built-in HIER_NORMAL law under the own
Philox stream, the same bits at every chunk width, bit-identical launch variants, checkpoint / resume
and the blob of the unflagged program refused, and a NaN term."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from oracle import oracle as orc
from tests import user_laws_theta as ut
from tests.parity import GpuSession, compare_histories
from tests.test_gpu_mala import _hier_theta0, _hier_updates

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = ut.G
P = G + 2
TOL = 1e-12


def _law(name, gradient, chunk=None):
    hand, fwd, Df, _, _ = ut.LAWS[name]
    src = fwd if gradient == "forward" else hand
    return em.DeviceLaw(src, P, Df(P), gradient=gradient, chunk=chunk, theta_term=True)


def _session(law, updates, X, th0, Cn, seed=0, **cfg):
    g = GpuSession(law, updates, X, th0, Cn, seed=seed, **cfg)
    g.ck(law.abi_attach(g.lib, g.h))
    return g


def _ups():
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.01]), [1])]


# ---- every kernel against extended precision ----------------------------------------------------------
# 3001 rows: S = 11 segments of about 272 rows under "chains" R = 1, the last one short; 7 rows: S = 1

CASES = [("hier", False, None), ("hier", True, None), ("hier", "forward", None), ("hier", "forward", 3),
         ("hier", "forward", 5), ("ridge", True, None), ("ridge", "forward", None), ("ridge", "forward", 3)]


@pytest.mark.parametrize("variant", [11, 12, 14, 2])
@pytest.mark.parametrize("name,gradient,chunk", CASES)
def test_every_kernel_against_extended_precision(name, gradient, chunk, variant):
    for N in (3001, 7):
        X = ut.data(name, N, P, seed=21)
        Cn = 701
        th = ut.theta(name, P, Cn, seed=22)
        law = _law(name, gradient, chunk)
        g = _session(law, _ups(), X, th, Cn, sweep_variant=variant)
        v = g.variant()
        assert v == "user_lanes" if variant == 2 else v.startswith("user_chains_R"), v
        ll_v = g.eval_loglik()
        llw, lla, grw, gra = ut.reference(name, th, X)
        e_ll = np.abs(ll_v - llw) / (TOL * lla)
        assert e_ll.max() <= 1, (N, v, e_ll.max())
        if gradient:
            ll_g, gr = g.eval_grad()
            assert np.array_equal(ll_g, ll_v) if gradient == "forward" else e_ll.max() <= 1
            e_g = np.abs(gr - grw) / (TOL * np.maximum(gra, 1e-300))
            print(f"{name} {gradient} K={law.chunk} N={N} {v}: grad err / tol {e_g.max():.3g}, ll {e_ll.max():.3g}")
            assert e_g.max() <= 1, (N, v, np.unravel_index(np.argmax(e_g), e_g.shape), e_g.max())
        assert g.lib.extmcmc_sync(g.h) == _abi.OK
        g.close()


def test_nan_term_rejects_without_a_domain_error():
    # log lambda = +inf: lambda / 2 |beta|^2 - (P - 1) / 2 log lambda is inf - inf
    X = ut.data("ridge", 500, P, seed=3)
    Cn = 64
    th = ut.theta("ridge", P, Cn, seed=4)
    bad = np.zeros(Cn, bool)
    bad[::5] = True
    th[P - 1, bad] = np.inf
    g = _session(_law("ridge", True), _ups(), X, th, Cn)
    ll, gr = g.eval_grad()
    assert g.lib.extmcmc_sync(g.h) == _abi.OK
    assert np.isnan(ll[bad]).all() and np.isfinite(ll[~bad]).all()
    # d/d log lambda = (P - 1) / 2 - lambda / 2 |beta|^2 = -inf there
    assert not np.isfinite(gr[P - 1, bad]).any() and np.isfinite(gr[:, ~bad]).all()
    # the proposal of such a state is rejected
    props = th[None, :1, :]          # coordinate 1 unchanged: the proposal is the state
    out = g.run(list(em.MCMCSchedule(1, 1)), replay=(props, np.random.default_rng(0).exponential(size=(1, Cn))))
    assert not out["accepted"][0, bad].any()
    g.close()


# ---- the hierarchical restatement against the built-in law -----------------------------------------------

@pytest.mark.parametrize("gradient", [True, "forward"])
@pytest.mark.parametrize("Cn,ragged", [(200, False), (7, True)])
def test_replay_parity_hier_restatement_cfg4(gradient, Cn, ragged):
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
    rep["variant"] = g.variant()
    if rep["chains_diverged"] == 0:
        so, sg = o.stats(), g.stats()
        rep["eps_bitexact"] = all(np.array_equal(o.eps(u), g.eps(u)) for u in range(1, len(ups) + 1))
        rep["moments_bitexact"] = bool(np.array_equal(so["mean"], sg["mean"]) and np.array_equal(so["cov"], sg["cov"]))
        rep["counts_equal"] = bool(np.array_equal(so["n_accept"], sg["n_accept"]))
    g.close()
    print(rep)
    assert rep["accept_mismatch"] == 0 and rep["theta_bitexact"] and rep["ll_rel_err"] < 1e-10, rep
    assert 0.02 < rep["accept_rate"] < 0.98, rep
    if rep["chains_diverged"] == 0:
        assert rep["eps_bitexact"] and rep["moments_bitexact"] and rep["counts_equal"], rep


def test_same_decisions_as_the_builtin_law_under_own_philox():
    X, grp = ut.hier_data(2000, seed=7, ragged=True)
    Cn, M = 512, 40
    ups = _hier_updates(G)
    th0 = _hier_theta0(G, Cn)
    steps = list(em.MCMCSchedule(M, len(ups)))
    gb = GpuSession(em.HierNormalLaw(G), ups, X[:, 0].copy(), th0, Cn, seed=7, n_steps_hint=len(steps), y=grp)
    rb = gb.run(steps)
    gu = _session(_law("hier", True), ups, X, th0, Cn, seed=7, n_steps_hint=len(steps))
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
    okt = np.broadcast_to(ok[:, None], rb["theta"].shape)
    # MALA moves along the gradient, which the two laws also sum in different orders: the states agree to
    # rounding, the decisions exactly
    assert np.allclose(rb["theta"][okt], ru["theta"][okt], rtol=1e-12, atol=1e-14)
    rel = np.abs(rb["ll_prop"] - ru["ll_prop"])[ok] / np.abs(rb["ll_prop"][ok])
    assert rel.max() < 1e-10
    assert near_ties <= Cn // 100
    assert 0.05 < rb["accepted"].mean() < 0.95
    gb.close(); gu.close()


# ---- forward mode: the same bits at every width -----------------------------------------------------------

PINNED = dict(sweep_variant=11)


def test_every_width_gives_the_same_bits():
    Cn = 701
    X = ut.data("hier", 3001, P, seed=41)
    th = ut.theta("hier", P, Cn, seed=42)
    ref = None
    for K in (None, 1, 3, P):
        g = _session(_law("hier", "forward", K), _ups(), X, th, Cn, **PINNED)
        ll_v = g.eval_loglik()
        ll, gr = g.eval_grad()
        assert g.variant() == "user_chains_R1"
        g.close()
        assert np.array_equal(ll, ll_v), K
        ref = ref or (ll, gr)
        assert np.array_equal(ll, ref[0]) and np.array_equal(gr, ref[1]), K


def test_mala_under_replay_is_bit_identical_across_widths():
    Cn, M = 256, 60
    X, grp = ut.hier_data(300, seed=8, ragged=True)
    ups = _hier_updates(G, tau=0.05)
    th0 = _hier_theta0(G, Cn)
    steps = list(em.MCMCSchedule(M, len(ups)))
    o = orc.Oracle(em.HierNormalLaw(G), ups, X[:, 0].copy(), th0, Cn, seed=4, y=grp)
    ro = o.run(steps, n_threads=8)
    runs = {}
    for K in (None, 1, 3, P):
        g = _session(_law("hier", "forward", K), ups, X, th0, Cn, seed=4, n_steps_hint=len(steps), **PINNED)
        runs[K] = g.run(steps, replay=(ro["proposals"], ro["exp_draws"]))
        g.close()
    ref = runs[None]
    assert 0.05 < ref["accepted"].mean() < 0.95, ref["accepted"].mean()
    for K in (1, 3, P):
        for key in ("theta", "ll", "accepted", "theta_prop", "ll_prop"):
            assert np.array_equal(runs[K][key], ref[key], equal_nan=True), (K, key)


# ---- determinism -----------------------------------------------------------------------------------------

_JOB = r"""
import json, sys, numpy as np
sys.path.insert(0, '.')
import extensiblemcmc_jl_b200 as em
from tests import user_laws_theta as ut
from tests.test_gpu_mala import _hier_theta0, _hier_updates
from tests.test_gpu_user_law_theta import _law, _session
G, P = ut.G, ut.G + 2
X, _ = ut.hier_data(300, seed=4, ragged=True)
th0 = _hier_theta0(G, 300)
steps = list(em.MCMCSchedule(12, 3))
out = {}
for gradient in (True, "forward"):
    for name, cfg, block, splits in [("eager_all", dict(use_graphs=0), 36, [(0, 300)]),
                                     ("graph_all", dict(use_graphs=1), 36, [(0, 300)]),
                                     ("graph_b4", dict(use_graphs=1), 4, [(0, 300)]),
                                     ("eager_b1", dict(use_graphs=0), 1, [(0, 300)]),
                                     ("split", dict(use_graphs=1), 36, [(0, 130), (130, 300)])]:
        th, ll = [], []
        for lo, hi in splits:
            g = _session(_law("hier", gradient), _hier_updates(G), X, np.ascontiguousarray(th0[:, lo:hi]), hi - lo,
                         seed=7, chain_offset=lo, n_steps_hint=36, **cfg)
            for b in range(0, len(steps), block):
                g.run(steps[b:b + block])
            t, l = g.state()
            th.append(t); ll.append(l)
            g.close()
        out[f"{gradient}_{name}"] = [np.concatenate(th, axis=1).tolist(), np.concatenate(ll).tolist()]
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
    for gradient in ("True", "forward"):
        ref = res[0][f"{gradient}_eager_all"]
        assert np.isfinite(np.array(ref[1])).all()
        assert not np.array_equal(np.array(ref[0]), _hier_theta0(G, 300))
        for out in res:
            for name, v in out.items():
                if name.startswith(gradient):
                    assert v == ref, name


def test_checkpoint_resume_and_the_unflagged_blob_is_refused():
    X, _ = ut.hier_data(200, seed=4)
    Cn, M = 150, 20
    ups = _hier_updates(G)
    th0 = _hier_theta0(G, Cn)
    s1 = list(em.MCMCSchedule(M, len(ups)))

    def save(g):
        n = C.c_int64()
        g.ck(g.lib.extmcmc_checkpoint_size(g.h, C.byref(n)))
        blob = (C.c_uint8 * n.value)()
        g.ck(g.lib.extmcmc_checkpoint_save(g.h, blob, n.value))
        return blob, n.value

    mk = lambda law, th: _session(law, ups, X, th, Cn, seed=5, n_steps_hint=2 * M)  # noqa: E731
    law = _law("hier", True)
    a = mk(law, th0)
    a.run(s1[:M]); a.run(s1[M:])
    th_a, ll_a = a.state()
    b = mk(law, th0)
    b.run(s1[:M])
    blob, n = save(b)
    c = mk(law, th0 * 0 + th0[:, :1])
    c.ck(c.lib.extmcmc_checkpoint_load(c.h, blob, n))
    c.seq = M
    c.run(s1[M:])
    th_c, ll_c = c.state()
    assert np.array_equal(th_a, th_c) and np.array_equal(ll_a, ll_c)
    # the same source compiled without the flag is another program, both ways
    plain = em.DeviceLaw(ut.HIER_HAND, P, 2, gradient=True)
    d = mk(plain, th0)
    assert d.lib.extmcmc_checkpoint_load(d.h, blob, n) == _abi.EINVAL
    assert b"another user law" in d.lib.extmcmc_last_error(d.h)
    d.run(s1[:M])
    blob_d, n_d = save(d)
    assert c.lib.extmcmc_checkpoint_load(c.h, blob_d, n_d) == _abi.EINVAL
    for s in (a, b, c, d):
        s.close()
