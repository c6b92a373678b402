"""Every kernel of the user-law sweep (csrc/sweep_user.cuh) against an extended-precision reference:
the "chains" mapping at R = 1 / 2 / 4 chains per thread and the "lanes" mapping, with and without the
gradient, forced and as the planner picks them.  Every chain is checked, the last CTA is ragged,
chains that share a theta column are bit-identical whichever R slot they sit in, odd obs_dim runs
over many tiles and segments, the 64 x 64 shape limit runs its spilling gradient kernels, and a
domain failure in one R slot stays in that slot.

The reference sums the per-row terms of tests/user_laws.py in np.longdouble (80-bit on x86-64):
|ll - ref| <= 1e-12 * sum|t| and |grad - ref| <= 1e-10 * sum|g|, per chain and coordinate."""
import ctypes as C
import functools

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws as ul
from tests.parity import theta_init_for
from tests.test_gpu_user_law import _data, _session, _theta

pytestmark = pytest.mark.gpu

LL_TOL, G_TOL = 1e-12, 1e-10
NT = 128                        # kUserNT: threads per CTA; chain slot r of thread t is cbase + r * NT + t
# every kernel user_law_load can fetch: extmcmc_user_{chains_r1,chains_r2,chains_r4,lanes}_g{0,1}
ALL_KERNELS = {f"{m}_g{g}" for m in ("chains_r1", "chains_r2", "chains_r4", "lanes") for g in (0, 1)}
_launched = set()               # kernels this module launched and checked
_variant_cases_done = []


def _rmax(P, grad):
    """user_max_R (sweep_user.cuh): chains per thread the "chains" mapping may hold."""
    n = 2 * P + 1 if grad else P + 1
    return 4 if 4 * n <= 40 else 2 if 2 * n <= 40 else 1


def _kernel(variant, grad):
    m = "lanes" if variant == "user_lanes" else "chains_r" + variant[len("user_chains_R"):]
    return f"{m}_g{1 if grad else 0}"


def _ups():
    # the sessions only evaluate: any update will do
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.01]), [1])]


def _reference(law, th, X, w=None, chunk=32):
    """Sum over rows of the per-row terms and gradients in np.longdouble, rows weighted by w (row
    multiplicities; None = 1): ll [C], sum|t| [C], grad [P, C], sum|g| [P, C], as float64."""
    terms = ul.LAWS[law][2]
    Cn = th.shape[1]
    wl = np.ones(len(X), np.longdouble) if w is None else np.asarray(w, np.longdouble)
    ll, lla = np.empty(Cn), np.empty(Cn)
    gr, gra = np.empty((th.shape[0], Cn)), np.empty((th.shape[0], Cn))
    for lo in range(0, Cn, chunk):
        t, g = terms(th[:, lo:lo + chunk], X, dtype=np.longdouble)
        ll[lo:lo + chunk] = (wl[:, None] * t).sum(axis=0)
        lla[lo:lo + chunk] = (wl[:, None] * np.abs(t)).sum(axis=0)
        gr[:, lo:lo + chunk] = (wl[None, :, None] * g).sum(axis=1)
        gra[:, lo:lo + chunk] = (wl[None, :, None] * np.abs(g)).sum(axis=1)
    return ll, lla, gr, gra


def _check(g, law, th, X, grad, ref=None, w=None, chains=None, tag=""):
    """eval_loglik (and eval_grad) of chains (default: every chain) against the reference; records
    the kernels launched.  Returns ll, grad."""
    ll = g.eval_loglik()
    v = g.variant()
    _launched.add(_kernel(v, False))
    gr = None
    if grad:
        ll_g, gr = g.eval_grad()
        _launched.add(_kernel(v, True))
        assert np.array_equal(ll_g, ll)
    assert g.lib.extmcmc_sync(g.h) == _abi.OK
    chains = np.arange(th.shape[1]) if chains is None else chains
    llw, lla, grw, gra = ref if ref is not None else _reference(law, th[:, chains], X, w)
    e_ll = np.abs(ll[chains] - llw) / (LL_TOL * lla)
    msg = f"{tag} {v}: ll err / tol {e_ll.max():.3g}"
    if grad:
        e_g = np.abs(gr[:, chains] - grw) / (G_TOL * np.maximum(gra, 1e-300))
        msg += f", grad err / tol {e_g.max():.3g}"
    print(msg)
    assert np.all(e_ll <= 1), (tag, v, chains[np.argmax(e_ll)], e_ll.max())
    if grad:
        assert np.all(e_g <= 1), (tag, v, np.unravel_index(np.argmax(e_g), e_g.shape), e_g.max())
    return ll, gr


# ---- every kernel, every chain ------------------------------------------------------------------

N_V = 3001                       # odd: the last tile reads the zero padding row
SHAPE_V = {"gsn1d": 1, "logistic": 9, "poisson_reg": 3}   # obs_dim of each law in the variant cases


def _dup_sets(Cn):
    """Chains that get one theta column: the R = 4 slots of thread 37 of the first CTA, the same
    thread of the second CTA, and the last (ragged) CTA's last chain."""
    return [c for c in (37, 37 + NT, 37 + 2 * NT, 37 + 3 * NT, 37 + 4 * NT, Cn - 1) if c < Cn] if Cn > 32 \
        else [3, 17, Cn - 1]


@functools.lru_cache(maxsize=None)
def _variant_problem(law, Cn):
    D = SHAPE_V[law]
    P = ul.LAWS[law][1](D)
    X = _data(law, N_V, D, seed=21)
    th = _theta(law, P, Cn, seed=22)
    dup = _dup_sets(Cn)
    th[:, dup] = th[:, dup[:1]]
    return X, th, dup, _reference(law, th, X)


# (sweep_variant, C): C = 701 leaves the last CTA ragged under every mapping (701 % 4, % 128, % 256
# and % 512 are non-zero); C = 29 forces the chains mapping where the planner picks lanes.
VARIANT_CASES = [(v, 701) for v in (0, 11, 12, 14, 2)] + [(v, 29) for v in (0, 1, 14)]


@pytest.mark.parametrize("grad", [False, True])
@pytest.mark.parametrize("variant,Cn", VARIANT_CASES)
@pytest.mark.parametrize("law", ["gsn1d", "logistic", "poisson_reg"])
def test_every_kernel_every_chain(law, variant, Cn, grad):
    D = SHAPE_V[law]
    P = ul.LAWS[law][1](D)
    X, th, dup, ref = _variant_problem(law, Cn)
    g = _session(ul.LAWS[law][0], grad, P, D, _ups(), X, th, Cn, sweep_variant=variant)
    rmax = _rmax(P, grad)
    v = g.variant()
    if variant in (11, 12, 14):
        assert v == f"user_chains_R{min(variant - 10, rmax)}", (v, rmax)
    elif variant == 2 or (variant == 0 and Cn <= 32):
        assert v == "user_lanes", v
    elif variant == 1 and Cn < NT:
        assert v == "user_chains_R1", v         # fewer chains than threads: no R > 1
    else:
        assert v.startswith("user_chains_R") and int(v[-1]) <= rmax, v
    ll, gr = _check(g, law, th, X, grad, ref=ref, tag=f"{law} D={D} C={Cn} sv={variant} grad={grad}")
    # one theta column in several R slots, CTAs and the ragged CTA: the same bits
    assert np.all(ll[dup] == ll[dup[0]]), ll[dup]
    if grad:
        assert np.all(gr[:, dup] == gr[:, dup[:1]]), gr[:, dup]
    g.close()
    _variant_cases_done.append((law, variant, Cn, grad))


def test_every_user_kernel_was_launched():
    n_cases = 3 * len(VARIANT_CASES) * 2
    if len(_variant_cases_done) < n_cases:
        pytest.skip("needs every case of test_every_kernel_every_chain in the same run")
    print("launched:", sorted(_launched))
    assert _launched == ALL_KERNELS, ALL_KERNELS - _launched


# ---- odd obs_dim over many tiles and segments ---------------------------------------------------

N_DEEP = 2**21 + 1               # odd; several segments of several tiles each (tile: 340 rows at D = 3)
POOL = 4096                      # distinct rows: the reference weighs each by its multiplicity


@pytest.mark.parametrize("variant,Cn", [(1, 150), (2, 7)])
@pytest.mark.parametrize("law,D", [("poisson_reg", 3), ("poisson_reg", 5), ("poisson_reg", 7),
                                   ("logistic", 3), ("logistic", 5)])
def test_odd_obs_dim_over_many_tiles_and_segments(law, D, variant, Cn):
    # D not a power of two: a tile (user_tile_rows(D) rows) is shorter than the stage, and tile
    # offsets are multiples of 2 D doubles.  The rows are drawn at random from a pool, so that a row
    # read twice, skipped or read from the wrong offset changes the sum.
    P = ul.LAWS[law][1](D)
    rng = np.random.default_rng(D)
    pool = _data(law, POOL, D, seed=30 + D)
    idx = rng.integers(0, POOL, N_DEEP)
    X = np.ascontiguousarray(pool[idx])
    th = _theta(law, P, Cn, seed=31)
    g = _session(ul.LAWS[law][0], True, P, D, _ups(), X, th, Cn, sweep_variant=variant)
    assert g.variant() == ("user_chains_R1" if variant == 1 else "user_lanes"), g.variant()
    _check(g, law, th, pool, True, w=np.bincount(idx, minlength=POOL), tag=f"{law} D={D} C={Cn} N={N_DEEP}")
    g.close()


# ---- the 64 x 64 shape limit ---------------------------------------------------------------------

@pytest.mark.parametrize("variant,Cn", [(1, 150), (2, 7)])
@pytest.mark.parametrize("law,D", [("poisson_reg", 64), ("logistic", 64)])
def test_shape_limit_64(law, D, variant, Cn):
    # the gradient kernels spill at this shape (P = 64: theta, Law and gradient do not fit the
    # register file); spilling costs time, never values
    P = ul.LAWS[law][1](D)
    N = 3001
    X = _data(law, N, D, seed=41)
    th = _theta(law, P, Cn, seed=42)
    g = _session(ul.LAWS[law][0], True, P, D, _ups(), X, th, Cn, sweep_variant=variant)
    assert g.variant() == ("user_chains_R1" if variant == 1 else "user_lanes"), g.variant()
    ll, gr = _check(g, law, th, X, True, tag=f"{law} P={P} D={D} C={Cn}")
    # central finite differences of the device's own log-likelihood, last chain (the ragged CTA)
    c = Cn - 1
    gra = _reference(law, th[:, c:], X)[3][:, 0]
    for k in range(P):
        h = 1e-6 * max(1.0, abs(th[k, c]))
        fd = []
        for s in (+1, -1):
            t2 = th.copy()
            t2[k, c] += s * h
            g.ck(g.lib.extmcmc_set_state(g.h, _abi.dptr(np.ascontiguousarray(t2))))
            fd.append(g.eval_loglik()[c])
        assert abs((fd[0] - fd[1]) / (2 * h) - gr[k, c]) <= 1e-5 * max(1.0, gra[k], abs(gr[k, c])), (k, fd, gr[k, c])
    g.close()


# ---- a domain failure in some R slots of one thread ------------------------------------------------

@pytest.mark.parametrize("variant", [14, 2])
def test_domain_failure_stays_in_its_slot(variant):
    Cn, N = 701, 2001
    X = _data("gsn1d", N, 1, seed=51)
    th = _theta("gsn1d", 2, Cn, seed=52)
    # under R = 4: thread 37 of CTA 0 holds 37, 165, 293, 421; thread 44 holds 44, ..., 300, 428;
    # threads 5 and 8 of the ragged CTA 1 hold 517, 645 and 520, 648
    bad = np.array([37, 300, 520, 645])
    th[1, bad] = [-1.0, np.inf, np.nan, 0.0]
    good = np.setdiff1d(np.arange(Cn), bad)
    g = _session(ul.GSN1D, True, 2, 1, _ups(), X, th, Cn, sweep_variant=variant)
    assert g.variant() == ("user_chains_R4" if variant == 14 else "user_lanes"), g.variant()
    ll = g.eval_loglik()
    assert g.lib.extmcmc_sync(g.h) == _abi.EDOMAIN
    assert g.lib.extmcmc_sync(g.h) == _abi.OK           # reported once
    ll_g, gr = g.eval_grad()
    assert g.lib.extmcmc_sync(g.h) == _abi.EDOMAIN
    assert np.array_equal(ll_g, ll, equal_nan=True)
    assert np.isnan(ll[bad]).all() and np.isnan(gr[:, bad]).all()
    assert np.isfinite(ll[good]).all() and np.isfinite(gr[:, good]).all()
    llw, lla, grw, gra = _reference("gsn1d", th[:, good], X)
    e_ll = np.abs(ll[good] - llw) / (LL_TOL * lla)
    e_g = np.abs(gr[:, good] - grw) / (G_TOL * gra)
    print(f"domain sv={variant} {g.variant()}: ll err / tol {e_ll.max():.3g}, grad err / tol {e_g.max():.3g}")
    assert e_ll.max() <= 1 and e_g.max() <= 1, (e_ll.max(), e_g.max())
    g.close()


# ---- the benchmark's shape ---------------------------------------------------------------------------

def test_full_size_against_sufficient_statistics():
    # C = 4096, N = 1e6 (tools/user_law_bench.py, cfg 2): the planner's own choice on a B200 is R = 4
    n, Cn = 1_000_000, 4096
    x = 1.5 + 2.0 * np.random.default_rng(2).standard_normal(n)
    th = theta_init_for(x, Cn)
    g = _session(ul.GSN1D, False, 2, 1, _ups(), x[:, None], th, Cn)
    assert g.variant() == "user_chains_R4", g.variant()
    ll = g.eval_loglik()
    assert g.lib.extmcmc_sync(g.h) == _abi.OK
    # sum_j [c0 - h (x_j - mu)^2] = N c0 - h (Sxx + N (xbar - mu)^2), in extended precision
    xl = x.astype(np.longdouble)
    xbar = xl.sum() / n
    sxx = ((xl - xbar) ** 2).sum()
    mu, var = th[0].astype(np.longdouble), th[1].astype(np.longdouble)
    want = n * (-(ul.LOG2PI + np.log(var)) / 2) - (sxx + n * (xbar - mu) ** 2) / (2 * var)
    # var > 1 / (2 pi): every term is negative, so sum|t| = |ll|
    assert (th[1] > 1 / (2 * np.pi)).all()
    e = np.abs(ll - want.astype(np.float64)) / (LL_TOL * np.abs(want.astype(np.float64)))
    print(f"full size {g.variant()}: ll err / tol {e.max():.3g}")
    assert e.max() <= 1, e.max()
    g.close()
