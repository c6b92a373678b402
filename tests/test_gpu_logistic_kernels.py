"""Every kernel of the logistic sweep (csrc/sweep_logistic.cu, DESIGN K4) against an extended-precision
reference: sweep_logistic_kernel<D, PM> at D = 32 / 64 / 128 / 256 and both phase-1 modes (PM = 2, the
default, and PM = 0, EXTMCMC_LOGI_PHASE1=0, run in a process of its own), on every chain and
coordinate, with d on both sides of every padding boundary and (n, C) chosen so that every case of the
flattened (chain block x tile) work split is taken; the softplus/sigmoid epilogue over |z| from 0 to
1e300 through the real kernel; and MALA replay parity against the oracle at cfg 3's parameter counts.

The reference forms z, ll and the gradient in np.longdouble (80-bit on x86-64).  With u = 2^-53,
a_i = sum_k |x_ik theta_k| and sigma' = sigma (1 - sigma), per chain and coordinate:

  |ll - ref|      <= TOL * sum_i (|y_i z_i| + softplus(z_i) + a_i)
  |grad_k - ref_k| <= TOL * sum_i |x_ik| (1 + sigma'(z_i) a_i),       TOL = 1e-13.

Derivation (first order; the bound is on the magnitudes of the operands, since with y = 1 and large z
a term y z - softplus(z) is a cancellation whose fp64 error is relative to |z|, not to the term):
- z: every accumulator chain of phase 1 takes D / 16 DMMAs of 4 products (PM = 2: four chains added
  pairwise; PM = 0: two half-range chains, their sum, then the partner's half), so even with one
  rounding per product |dz_i| <= (D/4 + 4) u a_i = gz a_i.
- ll: d(y z - sp)/dz = y - sigma lies in [-1, 1]; the epilogue adds 5.1e-16 sp (the softplus bound of
  the probe below) and one rounding of y z - sp.  A thread then adds one row per tile of its piece
  (T_p tiles), a 3-level shuffle tree, the pair add and at most S pieces in the finalize kernel:
  |dll| <= gz sum a + (5.1e-16 + (T_p + S + 5) u) sum (|y z| + sp).
- grad: |dr_i| <= sigma' gz a_i + 6.6e-16 + u (sigmoid bound, rounding of y - sg, |r| <= 1); phase 2
  accumulates the 16 T_p rows of a piece one product at a time at worst, then at most S pieces:
  |dg_k| <= sum_i |x_ik| (sigma' gz a_i + 6.6e-16 + (16 T_p + S + 1) u).
So TOL >= max(gz, 6.6e-16 + (16 T_p + S + 1) u) suffices; _derived_tol computes it from the mirror of
the work split for every shape, and every shape here keeps it below 1e-13 (gz = 7.5e-15 at D = 256).
Each bound is shown to discriminate on the data regime (a) shapes: dropping the last live row, adding
one zero-padded row (y = 0: -ln 2) or swapping two adjacent gradient rows falls outside it.

The softplus/sigmoid probe (one observation x = e_{d-1}, theta_{d-1,c} = z_c, so z is formed exactly):
relative error <= 5.1e-16 (softplus) and 6.6e-16 (sigmoid) for z >= -700 (DESIGN K4: 5.0e-16 and
6.5e-16 on a host replica); below -700 the documented clamp returns exp(-700) for exp(z), an absolute
error under exp(-700) < 1e-304.  With y = 1 the errors are absolute and allow the one rounding of
z - sp and 1 - sg (|z - sp| <= |z| + sp, |1 - sg| <= 1): u (|z| + sp) + 5.1e-16 sp and u + 6.6e-16 sigma."""
import functools
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests.parity import GpuSession, replay_compare

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LD = np.longdouble
U53 = 2.0 ** -53
TOL = 1e-13
SP_REL, SG_REL, CLAMP_ABS = 5.1e-16, 6.6e-16, 1e-304
KBM, KBN = 16, 64                # observations per tile, chains per block (sweep_logistic.cu)
# 8 fragment slots 8 w8 + 2 tq + e of one chain block: every w8, every tq, both e, and (phase 2:
# chain 8 w8 + gq) every gq
SLOTS = [0, 9, 18, 27, 36, 45, 54, 63]

_checked = set()                 # (D, phase-1 mode) pairs launched and checked
_cases_done = []
_worst = {}                      # part -> largest error / bound
_mode_bits = {}                  # case -> modes 0 and 2 agree bit for bit


def _note(part, r):
    _worst[part] = max(_worst.get(part, 0.0), float(r))


# ---- mirror of the planner (plan_sweep_logistic, unit_lo, cta_of_unit, logistic_padded_dim) ---------

def padded_dim(d):
    for D in (32, 64, 128, 256):
        if d <= D:
            return D
    return 0


def unit_lo(c, U, n_cta):
    return c * U // n_cta


def cta_of_unit(x, U, n_cta):
    c = x * n_cta // U
    while c + 1 < n_cta and unit_lo(c + 1, U, n_cta) <= x:
        c += 1
    while c > 0 and unit_lo(c, U, n_cta) > x:
        c -= 1
    return c


def split(n, Cn, sms):
    """The work split of one sweep: blocks, tiles per block T, units U, CTAs, partial slots S, the
    number of pieces of every block, the longest piece (tiles) and whether a CTA straddles blocks."""
    groups, T = -(-Cn // KBN), -(-n // KBM)
    U = groups * T
    n_cta = min(U, sms)
    S = -(-n_cta // groups) + 1
    npieces = [cta_of_unit((b + 1) * T - 1, U, n_cta) - cta_of_unit(b * T, U, n_cta) + 1 for b in range(groups)]
    tp, straddle = 0, False
    for c in range(n_cta):
        u, hi = unit_lo(c, U, n_cta), unit_lo(c + 1, U, n_cta)
        straddle |= hi > u and u // T != (hi - 1) // T
        while u < hi:
            m = min(T - u % T, hi - u)
            tp, u = max(tp, m), u + m
    return dict(groups=groups, T=T, U=U, n_cta=n_cta, S=S, npieces=npieces, tp=tp, straddle=straddle)


def _derived_tol(d, n, Cn, sms):
    s = split(n, Cn, sms)
    gz = (padded_dim(d) / 4 + 4) * U53
    return max(gz, SP_REL + (s["tp"] + s["S"] + 5) * U53, SG_REL + (16 * s["tp"] + s["S"] + 1) * U53)


def _hits(tag, s, sms):
    return {"U<SMs": s["U"] < sms and s["n_cta"] == s["U"] and s["tp"] == 1,
            "blocks>SMs": s["groups"] > sms,
            "spread": s["groups"] == 1 and s["npieces"][0] == sms,
            "straddle": s["straddle"],
            "slotS-1": max(s["npieces"]) == s["S"]}[tag]


# ---- the cases ---------------------------------------------------------------------------------------

def _fixed(n, Cn):
    return lambda sms: (n, Cn)


def _searched(tags, groups, tiles, n_of_T, C_of_groups):
    """(n, C) of the first (blocks, tiles per block) at which the split on `sms` SMs takes every case
    in `tags`: block-count and tile-count boundaries fall differently for every SM count."""
    def shape(sms):
        for g in groups(sms):
            for T in tiles:
                n, Cn = n_of_T(T), C_of_groups(g)
                s = split(n, Cn, sms)
                if all(_hits(t, s, sms) for t in tags):
                    return n, Cn
        raise AssertionError(f"no shape takes {tags} on {sms} SMs")
    return shape


# (name, d, (n, C) of the SM count, regime, tags).  Regimes: a = X / sqrt(d), theta near beta;
# b = theta x 200 (|z| in the hundreds, past +-700); c = column scales 10^U(-3, 3), all-zero rows and
# columns; y0 / y1 = regime a with y all 0 / all 1.  The fixed "U<SMs" shapes have at most 126 units
# and so need more than 126 SMs (a B200 has 148); the shapes of the other cases are searched for the
# device's SM count (on 148 SMs: d33 C = 9605, d100 n = 2049 C = 130, d129 n = 1179 C = 261).
CASES = [
    ("d1", 1, _fixed(333, 1), "y1", ["U<SMs"]),
    ("d31", 31, _fixed(15, 63), "a", ["U<SMs"]),
    ("d32", 32, _fixed(16, 64), "b", ["U<SMs"]),
    ("d33", 33, _searched(["blocks>SMs", "straddle"], lambda s: range(s + 3, s + 40), [2],
                          lambda T: 17, lambda g: KBN * (g - 1) + 5), "c", ["blocks>SMs", "straddle"]),
    ("d63", 63, _fixed(1000, 65), "a", ["U<SMs"]),
    ("d64", 64, lambda s: (KBM * 2 * s + 9, 7), "a", ["spread"]),
    ("d65", 65, _fixed(17, 65), "y0", ["U<SMs"]),
    ("d100", 100, _searched(["straddle"], lambda s: (3, 5, 7), range(129, 400),
                            lambda T: KBM * T - 15, lambda g: KBN * (g - 1) + 2), "a", ["straddle"]),
    ("d127", 127, _fixed(999, 7), "b", ["U<SMs"]),
    ("d128", 128, _fixed(777, 100), "c", ["U<SMs"]),
    ("d129", 129, _searched(["slotS-1", "straddle"], lambda s: (5, 7, 9, 11, 13), range(60, 400),
                            lambda T: KBM * T - 5, lambda g: KBN * (g - 1) + 5), "a", ["slotS-1", "straddle"]),
    ("d200", 200, _fixed(600, 70), "b", ["U<SMs"]),
    ("d255", 255, _fixed(1, 65), "c", ["U<SMs"]),
    ("d256", 256, _fixed(837, 150), "a", []),
]
CASE = {c[0]: c for c in CASES}


def _shape(name, sms):
    _, d, shape, regime, tags = CASE[name]
    return (d,) + shape(sms) + (regime, tags)


@functools.lru_cache(maxsize=None)
def _case_data(name, sms):
    d, n, Cn, regime, _ = _shape(name, sms)
    rng = np.random.default_rng(100 + list(CASE).index(name))
    X = rng.standard_normal((n, d)) / math.sqrt(d)
    beta = rng.standard_normal(d)
    th = beta[:, None] + 0.3 * rng.standard_normal((d, Cn))
    if regime == "c":
        scale = 10.0 ** rng.uniform(-3, 3, d)
        X *= scale * math.sqrt(d)
        beta /= scale * math.sqrt(d)
        th /= (scale * math.sqrt(d))[:, None]
        X[3::7] = 0.0                               # z = 0 exactly: sp = ln 2, r = y - 1/2
        if d >= 3:
            X[:, [0, d // 2]] = 0.0                 # their gradient rows must be exactly 0
    y = (rng.random(n) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
    if regime == "b":
        th *= 200.0
    elif regime in ("y0", "y1"):
        y[:] = 0.0 if regime == "y0" else 1.0
    if Cn >= KBN:
        th[:, SLOTS] = th[:, :1]
    return X, y, np.ascontiguousarray(th)


def _softplus_sigmoid(z):
    e = np.exp(-np.abs(z))
    return np.maximum(z, 0) + np.log1p(e), np.where(z >= 0, 1 / (1 + e), e / (1 + e))


@functools.lru_cache(maxsize=None)
def _reference(name, sms):
    """ll, grad (np.longdouble), their bounds (TOL x operand magnitudes) and the last live row's
    term of every chain."""
    X, y, th = _case_data(name, sms)
    n, d = X.shape
    Cn = th.shape[1]
    Xl, yl, Xa = X.astype(LD), y.astype(LD)[:, None], np.abs(X)
    ll, gr = np.empty(Cn, LD), np.empty((d, Cn), LD)
    ll_tol, gr_tol, t_last = np.empty(Cn), np.empty((d, Cn)), np.empty(Cn)
    chunk = max(1, 2_000_000 // n)
    for lo in range(0, Cn, chunk):
        sl = slice(lo, lo + chunk)
        Z = Xl @ th[:, sl].astype(LD)
        sp, sg = _softplus_sigmoid(Z)
        t = yl * Z - sp
        ll[sl] = t.sum(axis=0)
        t_last[sl] = t[-1]
        gr[:, sl] = Xl.T @ (yl - sg)
        A = Xa @ np.abs(th[:, sl])
        ll_tol[sl] = TOL * (np.abs(yl * Z) + sp + A).sum(axis=0).astype(np.float64)
        s1 = (sg * (1 - sg)).astype(np.float64)
        gr_tol[:, sl] = TOL * (Xa.T @ (1.0 + s1 * A))
    return ll, gr, ll_tol, gr_tol, t_last


# ---- device runs ---------------------------------------------------------------------------------------

def _ups():
    # the sessions only evaluate: any update will do
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.01]), [1])]


def run_case(name, sms):
    """One session: eval_grad, eval_loglik twice; the arrays the checks need."""
    X, y, th = _case_data(name, sms)
    d, Cn = th.shape
    g = GpuSession(em.LogisticLaw(d), _ups(), X, th, Cn, y=y)
    try:
        assert g.variant() == "logistic_dmma", g.variant()
        ll, gr = g.eval_grad()
        ll1, ll2 = g.eval_loglik(), g.eval_loglik()
        assert g.lib.extmcmc_sync(g.h) == _abi.OK
    finally:
        g.close()
    return dict(ll=ll, gr=gr, ll_loglik=ll1, ll_again=ll2, shape=np.array([d, X.shape[0], Cn]))


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def sms():
    return _sms()


_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, %r)
from tests import test_gpu_logistic_kernels as m
sms, out = int(sys.argv[1]), sys.argv[2]
arrs = {}
for name in m.CASE:
    for k, v in m.run_case(name, sms).items():
        arrs[name + ":" + k] = v
np.savez(out, **arrs)
print("done", len(arrs))
""" % ROOT


@pytest.fixture(scope="module")
def mode0_results(sms, tmp_path_factory):
    """Every case under EXTMCMC_LOGI_PHASE1=0 (read once per process: a child process of its own)."""
    out = str(tmp_path_factory.mktemp("logi_pm0") / "pm0.npz")
    env = dict(os.environ, EXTMCMC_LOGI_PHASE1="0")
    r = subprocess.run([sys.executable, "-c", _CHILD, str(sms), out], capture_output=True, text=True,
                       timeout=900, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    z = np.load(out)
    return {name: {k: z[name + ":" + k] for k in ("ll", "gr", "ll_loglik", "ll_again", "shape")} for name in CASE}


_mode2 = {}


def _check_case(name, sms, res, mode):
    d, n, Cn, regime, tags = _shape(name, sms)
    assert list(res["shape"]) == [d, n, Cn]
    s = split(n, Cn, sms)
    assert max(s["npieces"]) <= s["S"], s                # the slots plan_sweep_logistic reserves
    for tag in tags:
        assert _hits(tag, s, sms), (name, tag, {k: v for k, v in s.items() if k != "npieces"})
    assert _derived_tol(d, n, Cn, sms) <= TOL, (name, _derived_tol(d, n, Cn, sms))
    ll, gr = res["ll"], res["gr"]
    # eval_loglik returns eval_grad's ll bits, and again on a second evaluation
    assert np.array_equal(res["ll_loglik"], ll) and np.array_equal(res["ll_again"], ll)
    llr, grr, ll_tol, gr_tol, t_last = _reference(name, sms)
    e_ll = np.abs(ll.astype(LD) - llr).astype(np.float64) / ll_tol
    err_g = np.abs(gr.astype(LD) - grr).astype(np.float64)
    assert np.all(err_g[gr_tol == 0] == 0)               # all-zero columns: exactly 0
    e_g = err_g / np.where(gr_tol > 0, gr_tol, 1.0)
    print(f"{name} D={padded_dim(d)} PM={mode} n={n} C={Cn} ({regime}): ll err / tol {e_ll.max():.3g}, "
          f"grad err / tol {e_g.max():.3g}")
    assert np.all(e_ll <= 1), (name, mode, int(np.argmax(e_ll)), e_ll.max())
    assert np.all(e_g <= 1), (name, mode, np.unravel_index(np.argmax(e_g), e_g.shape), e_g.max())
    _note("every chain: ll", e_ll.max())
    _note("every chain: grad", e_g.max())
    # one theta column in 8 fragment slots of block 0: the same bits
    if Cn >= KBN:
        assert np.all(ll[SLOTS] == ll[0]), ll[SLOTS]
        assert np.all(gr[:, SLOTS] == gr[:, :1]), name
    if regime == "a":
        # the bounds discriminate: a dropped last row, one zero-padded row counted (y = 0, z = 0:
        # -ln 2) and two adjacent gradient rows swapped all fall outside them
        assert np.all(np.abs(t_last) > ll_tol), name
        assert np.all(math.log(2) > ll_tol), name
        sw = np.abs(grr[d - 1] - grr[d - 2]).astype(np.float64)
        assert np.any(sw > gr_tol[d - 2]) and np.any(sw > gr_tol[d - 1]), name


@pytest.mark.parametrize("name", list(CASE))
def test_every_chain_phase1_default(name, sms):
    res = run_case(name, sms)
    _check_case(name, sms, res, 2)
    _mode2[name] = res
    _checked.add((padded_dim(CASE[name][1]), 2))
    _cases_done.append((name, 2))


@pytest.mark.parametrize("name", list(CASE))
def test_every_chain_phase1_pair_exchange(name, sms, mode0_results):
    res = mode0_results[name]
    _check_case(name, sms, res, 0)
    if name in _mode2:
        _mode_bits[name] = bool(np.array_equal(res["ll"], _mode2[name]["ll"]) and
                                np.array_equal(res["gr"], _mode2[name]["gr"]))
    _checked.add((padded_dim(CASE[name][1]), 0))
    _cases_done.append((name, 0))


def test_every_instantiation_was_checked():
    if len(_cases_done) < 2 * len(CASES):
        pytest.skip("needs every case of both phase-1 modes in the same run")
    print("checked (D, phase-1 mode):", sorted(_checked))
    print("modes 0 and 2 bit-identical:", json.dumps(_mode_bits))
    print("largest error / bound:", json.dumps(_worst))
    assert _checked == {(D, m) for D in (32, 64, 128, 256) for m in (0, 2)}
    # mode 0 adds z as (za + zb) + partner's half against mode 2's (zc0 + zc1) + (zc2 + zc3): the
    # results agree to the bounds above, not bit for bit (which also shows the child ran PM = 0)
    assert not all(_mode_bits.values()), _mode_bits


def test_unsupported_dimension_is_refused():
    d = 257
    X, y = np.zeros((16, d)), np.zeros(16)
    with pytest.raises(_abi.ExtMCMCError) as ei:
        GpuSession(em.LogisticLaw(d), _ups(), X, np.zeros(d), 4, y=y)
    assert ei.value.code == _abi.EUNSUPPORTED
    assert "LOGISTIC needs obs_dim = n_params = d with 1 <= d <= 256" in str(ei.value)


# ---- softplus / sigmoid through the real kernel ----------------------------------------------------------

PROBE_C = 64 * 512


def _ulps(b, k):
    """b (> 0) moved by -k .. k ulps."""
    bits = np.asarray(b, np.float64).view(np.int64)
    return np.concatenate([(bits + j).view(np.float64) for j in range(-k, k + 1)])


def probe_z():
    ln2 = math.log(2)
    # e = 2^-52, 2^-54, the clamp, the smallest normal / largest finite exp, the smallest subnormal
    edges = np.array([52 * ln2, 54 * ln2, 700.0, 1022 * ln2, math.log(np.finfo(np.float64).max), 745.1332191019411])
    # k of the exponent reduction: every one up to 63, then spread up to |z| = 745
    ks = np.unique(np.r_[np.arange(64), np.geomspace(64, 34400, 560).astype(np.int64)])
    mags = [np.logspace(-300, 300, 2000),
            _ulps(np.log(128.0 / np.arange(1, 128)), 3),          # 1 + e at a reciprocal-table boundary
            _ulps((ks + 0.5) * ln2 / 32, 3),                       # rounding boundaries of rint(x 32/ln2)
            _ulps(edges, 8),
            (edges[:, None] + np.linspace(-0.01, 0.01, 21)).ravel()]
    m = np.concatenate(mags)     # j = 128 (1 + e = 2, idx = 127) is z = 0 +- ulps below
    z = np.concatenate([[0.0, -0.0, 5e-324, -5e-324, 1e-323, -1e-323], m, -m, np.linspace(-720, 720, 16001)])
    assert z.size <= PROBE_C, z.size
    rest = np.random.default_rng(7).uniform(-40, 40, PROBE_C - z.size)
    return np.concatenate([z, rest])


@pytest.mark.parametrize("d", [1, 33, 65, 129])
def test_softplus_sigmoid_probe(d):
    z = probe_z()
    X = np.zeros((1, d))
    X[0, d - 1] = 1.0
    th = np.zeros((d, PROBE_C))
    th[d - 1] = z
    g = GpuSession(em.LogisticLaw(d), _ups(), X, th, PROBE_C, y=np.zeros(1))
    out = {}
    for yv in (0.0, 1.0):
        g.ck(g.lib.extmcmc_upload_obs(g.h, _abi.dptr(X), 1, d, _abi.dptr(np.array([yv]))))
        out[yv] = g.eval_grad()
    g.close()
    zl = z.astype(LD)
    spr, sgr = _softplus_sigmoid(zl)
    inner, clamped = z >= -700, z < -700
    assert clamped.any() and (z > 700).any()
    for yv, (ll, gr) in out.items():
        # the last feature lands in its own row; every other row is exactly 0
        assert np.all(gr[:d - 1] == 0.0), (d, yv)
        if yv == 0.0:
            err_sp, err_sg = np.abs(-ll.astype(LD) - spr), np.abs(-gr[d - 1].astype(LD) - sgr)
            tol_sp = np.where(inner, SP_REL * spr, CLAMP_ABS)
            tol_sg = np.where(inner, SG_REL * sgr, CLAMP_ABS)
        else:
            err_sp, err_sg = np.abs(ll.astype(LD) - (zl - spr)), np.abs(gr[d - 1].astype(LD) - (1 - sgr))
            tol_sp = U53 * (np.abs(zl) + spr) + np.where(inner, SP_REL * spr, CLAMP_ABS)
            tol_sg = U53 + np.where(inner, SG_REL * sgr, CLAMP_ABS)
        r_sp, r_sg = (err_sp / tol_sp).astype(np.float64), (err_sg / tol_sg).astype(np.float64)
        rel_sp = (err_sp[inner] / spr[inner]).max() if yv == 0.0 else float("nan")
        rel_sg = (err_sg[inner] / sgr[inner]).max() if yv == 0.0 else float("nan")
        print(f"probe d={d} D={padded_dim(d)} y={yv:g}: softplus err / bound {r_sp.max():.3g} (rel {float(rel_sp):.3g}), "
              f"sigmoid err / bound {r_sg.max():.3g} (rel {float(rel_sg):.3g})")
        assert np.all(r_sp <= 1), (d, yv, z[np.argmax(r_sp)], r_sp.max())
        assert np.all(r_sg <= 1), (d, yv, z[np.argmax(r_sg)], r_sg.max())
        _note("probe: softplus", r_sp.max())
        _note("probe: sigmoid", r_sg.max())


# ---- MALA replay parity at cfg 3's parameter counts -----------------------------------------------------

@pytest.mark.parametrize("d,n,Cn,iters,block,tau", [(100, 1500, 96, 30, 7, 0.4), (256, 600, 70, 20, None, 0.6)])
def test_mala_replay_parity_cfg3_dims(d, n, Cn, iters, block, tau):
    rng = np.random.default_rng(d)
    X = rng.standard_normal((n, d)) / math.sqrt(d)
    beta = rng.standard_normal(d)
    y = (rng.random(n) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
    th0 = 0.01 * rng.standard_normal((d, Cn))
    ups = [em.MALAUpdate(tau, list(range(1, d + 1)), prior=em.StandardPrior(em.Normal(0.0, 10.0)),
                         adpt=em.AdaptationMALA(adapt_every_k_steps=5, scale=0.01, offset=1.0))]
    # stats_mode 1 (running mean + variances) is what the front end picks for p > 16, cfg 3 included,
    # and it takes other step-kernel branches than the full covariance
    rep = replay_compare(X, Cn, iters, seed=3, updates=ups, law=em.LogisticLaw(d), y=y, theta_init=th0,
                         block=block, history_window=32, stats_mode=1)
    print(f"replay d={d}: ll rel err {rep['ll_rel_err']:.3g}, accept rate {rep['accept_rate']:.3f}")
    assert rep["variant"] == "logistic_dmma"
    assert rep["accept_mismatch"] == 0 and rep["near_ties"] == 0, rep
    assert rep["theta_bitexact"] and rep["ll_rel_err"] < 1e-10, rep
    assert rep["eps_bitexact"] and rep["counts_equal"] and rep["final_state_bitexact"], rep
    assert rep["mean_bitexact"] and rep["cov_bitexact"], rep      # variances: the oracle's diagonal
    assert 0.05 < rep["accept_rate"] < 0.98, rep
    _note("replay: ll rel err / 1e-10", rep["ll_rel_err"] / 1e-10)
