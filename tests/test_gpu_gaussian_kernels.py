"""Every kernel of the Gaussian sweeps (csrc/sweep_gsn1d.cu, DESIGN K2; csrc/sweep_gsnmv.cu, DESIGN K2')
against an extended-precision reference: sweep_gsn1d_chains_kernel<R> at R = 1 / 2 / 4 / 8 and
sweep_gsn1d_obs_kernel<CB> at CB = 1 ... 32, each without (eval_loglik) and with (eval_grad) the
first-order sums, for GsnTargetLaw([0.0]) and HierNormalLaw(G); sweep_gsnmv at d = 2 ... 16 under both
mappings.  Every chain and every group is checked; the shapes are chosen (searched, where the SM count
decides) so that every case of the planners is taken: S = 1, the max_S clamp, the cost search moving S
off its target, R falling back because the thread tiles would be mostly empty, a ragged last chain
group, empty segments in short groups, segments one observation past and short of a tile, odd tails
(the bulk copy reads the zero padding element), chain counts at 128 R +- 1, G on both sides of the
cooperative finish (kCoopG = 16), the fused tail against the separate reduction, and the L2
evict_first copy at an observation count twice the size at which it is switched on.

The reference works in np.longdouble (64-bit significand on x86-64, v = 2^-64) from centred sufficient
statistics of every group: with m the group's mean, A1 = sum (x - m), A2 = sum (x - m)^2 and
delta = m - mu, S = A2 + 2 delta A1 + n delta^2 and T = A1 + n delta.  Its own error is at most
(40 + log2 n) v M2 for S and (40 + log2 n) v M1 for T (pairwise sums of n terms, rounding of x - m and of
the combination), with M2 = A2 + 2 |delta A1| + n delta^2 >= sum (x - mu)^2 and
M1 = sum |x - m| + n |delta| >= sum |x - mu|; it is part of every bound below.

Kernel bounds, first order in u = 2^-53 (every bound is multiplied by 1.01 for the second-order terms):
- One term: x - mu is rounded once (relative u) and squared by an FMA into the accumulator, so the
  square carries 2u and every add u of the partial sum it makes.  S and T are sums of terms of one
  sign (S) or of magnitude |x - mu| (T); whatever the order, a sum whose longest path from a term to
  the result has k adds is off by at most k u sum |term|.  The longest path is
    * the per-thread chain: the segment length L for "chains" (one FMA per observation);
      2 ceil(L / 512) + 3 for "obs" (4 pairs per thread and full tile, one pair per thread of the
      partial tile, thread 0 takes the odd tail), then 5 shuffle levels and 8 warps;
    * the reduction of the S segment rows (G S for the hierarchical law): reduce_segments after
      eval_loglik, ceil(rows / 8) + 8 (8 slices) or rows (<= 16 rows); the fused tail of the "obs"
      mapping, ceil(rows / NS) + NS with NS = 256 / CB slices; grad_finalize_chain / _coop, S per
      group and then G groups.
  So |dS| <= (k + 3) u M2 and |dT| <= (k + 1) u M1.
- GsnTargetLaw(d = 1): ll = N c0 - S / (2 s2) with c0 = -(log 2pi + 2 log sqrt s2) / 2:
  |dc0| <= 4u (1 + log(2pi) / 2 + |log s2| / 2), |dll| <= N |dc0| + 2u N |c0| + (|dS| + 3u S) / (2 s2);
  d/dmu = T / s2: |d| <= (|dT| + u |T|) / s2; d/ds2 = -N / (2 s2) + S / (2 s2^2):
  |d| <= 2u N / (2 s2) + (|dS| + 4u S) / (2 s2^2).  Where the reference lies beyond the double range
  (s2 = 1e-200: S / (2 s2^2) ~ 1e405) the kernel must return the infinity of the same sign.
- HierNormalLaw: ll = -N log(2pi) / 2 - S / 2 + G (-log(2pi) / 2 - log tau) - D2 / (2 tau^2), D2 = sum_g dv_g^2,
  dv_g = th_g - mu: |dll| <= |dS| / 2 + (G + 10) u (N log(2pi) / 2 + S / 2 + G (1 + |log tau|) + D2 / (2 tau^2));
  d/dth_g = T_g - dv_g / tau^2: |d| <= |dT_g| + u |T_g| + 6u |dv_g| / tau^2;
  d/dmu = sum_g dv_g / tau^2: (G + 4) u sum_g |dv_g| / tau^2;
  d/dtau = -G / tau + D2 / tau^3: 2u G / tau + (G + 6) u D2 / tau^3.
- sweep_gsnmv: law_prepare factors Sigma = L L' (upper triangle only) and inverts L by forward
  substitution; with K = || |W| |L| ||_2 of the reference factor and g_n = n u / (1 - n u), the fp64
  factor and inverse change every quadratic form |W e|^2 by at most (g_{d+1} + 2 g_d) K^2 relative
  (backward errors |E| <= g_{d+1} |L||L'| of the factorisation and |F| <= g_d |L||W| of the inverse,
  both mapped through W), the rounding of x - mu and the row FMAs by 2 (g_d + u) K, the sum of squares
  by (d + 1) u: eps_q = (g_{d+1} + 2 g_d) K^2 + 2 (g_d + u) K + (d + 1) u per observation, so
  |dS| <= (eps_q + (k + 1) u) S with k as above (chains: L; obs: ceil(L / NT) + 5 + NT / 32, NT = 128
  for d <= 8 and 64 above).  logdet moves by at most g_{d+1} d K^2 / 2 through the factor, and
  |dll| <= N |dc0| + 2u N |c0| + |dS| / 2 + u S / 2.  The same formula covers the case with
  cond(Sigma) ~ 1e8 (K ~ 1e3 .. 1e4 there).  The reference's sums of n d-vectors use plain dot
  products: (n + 8d + 40) v ||W||_F^2 sum |x - mu|^2.

Each bound is shown to discriminate on the data regime (a) shapes (tests/test_gaussian_bounds.py, on
the host): dropping the last observation of the data or of a group, counting one zero padding element,
moving one observation to the neighbouring group, taking the neighbouring chain's T, and for gsnmv
using W' in place of W or the lower triangle in place of the upper one all fall outside the bound of
at least one output on every chain.

A known limit, not exercised: d/ds2 of GsnTargetLaw forms 2 s2 s2, which leaves the normal range for
s2 < 1.5e-154 (or > 1.3e154) even where the derivative itself is representable."""
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
from tests.parity import GpuSession

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LD = np.longdouble
U53 = 2.0 ** -53
V64 = LD(2) ** -64
SAFETY = 1.01
LOG2PI = np.log(LD(2) * np.arccos(LD(-1)))
CH_NT, CH_TILE = 128, 1024           # "chains" mapping of the 1-D sweep (sweep_gsn1d.cu)
OBS_NT, OBS_TILE = 256, 2048         # "obs" mapping
CB_ALL, R_ALL = (1, 2, 4, 8, 16, 32), (1, 2, 4, 8)

_checked = set()                     # instantiations launched and checked
_worst = {}                          # part -> largest error / bound


def _note(part, r):
    _worst[part] = max(_worst.get(part, 0.0), float(r))


# ---- mirror of the planners (plan_sweep_gsn1d, plan_sweep_gsnmv, segment_bounds) ------------------------

def _cdiv(a, b):
    return -(-a // b)


def chains_ctas_per_sm():
    """EXTMCMC_CHAINS_CTAS as the library reads it (atoi; <= 0 or unset: 8)."""
    e = os.environ.get("EXTMCMC_CHAINS_CTAS", "")
    digits = e.strip().lstrip("+")
    n = int(digits) if digits.isdigit() else 0
    return n if n > 0 else 8


def plan_gsn1d(C, n_largest, force, sms, G=1):
    n_pairs = (n_largest + 1) // 2
    chains, force_R = C > 32, 0
    if force > 10:
        force_R, force = force - 10, 1
    if force == 1:
        chains = True
    if force == 2 and C <= 32:
        chains = False
    if not chains:
        CB = 1
        while CB < C and CB < 32:
            CB <<= 1
        target, max_S = _cdiv(sms * 3, G), _cdiv(n_pairs, 1024)
        S = max(min(target, max_S), 1)
        return dict(kind="obs", R=CB, groups=1, S=S, G=G, target=target, max_S=max_S, clamped=S, trace=[],
                    name=f"gsn1d_obs_C{CB}")
    max_S, ctas, R, trace = _cdiv(n_pairs, 128), chains_ctas_per_sm(), 8, []
    while True:
        groups = _cdiv(C, CH_NT * R)
        target = _cdiv(sms * ctas, groups * G)
        S = clamped = max(min(target, max_S), 1)

        def cost(s):
            return _cdiv(groups * G * s, sms) * (_cdiv(n_pairs, s) + 32)
        best = S
        for s in range(S - 3 if S > 3 else 1, min(S + 3, max_S) + 1):
            if cost(s) < cost(best):
                best = s
        S = best
        fits, enough = C >= CH_NT * R, groups * S * G >= 2 * sms
        trace.append((R, fits, enough))
        if (R == force_R) if force_R else (R == 1 or (fits and enough)):
            break
        if R == 1:
            break
        R >>= 1
    return dict(kind="chains", R=R, groups=groups, S=S, G=G, target=target, max_S=max_S, clamped=clamped,
                trace=trace, name=f"gsn1d_chains_R{R}")


def plan_gsnmv(d, C, n, force, sms):
    chains = C > 32
    if force == 1:
        chains = True
    if force == 2 and C <= 65535:
        chains = False
    nt = 64 if d > 8 else 128
    groups = _cdiv(C, nt) if chains else C
    max_S = _cdiv((n + 1) // 2, 128)
    S = max(min(_cdiv(sms * 4, groups), max_S), 1)
    return dict(kind="chains" if chains else "obs", NT=nt, groups=groups, S=S, tile=(1024 // d) & ~1,
                name="gsnmv_chains" if chains else "gsnmv_obs")


def segments(n, S):
    """Lengths of the S segments of n observations (boundaries on even indices)."""
    P = (n + 1) // 2
    return [min(2 * ((s + 1) * P // S), n) - 2 * (s * P // S) for s in range(S)]


def thread_chain(plan, L):
    """Adds on the longest path of one segment of L observations up to the segment's row."""
    if plan["kind"] == "chains":
        return L
    if "NT" in plan:                                      # gsnmv "obs"
        return _cdiv(L, plan["NT"]) + 5 + plan["NT"] // 32
    return 2 * _cdiv(L, 2 * OBS_NT) + 3 + 5 + OBS_NT // 32


def reduce_depth(plan, path, G=1):
    rows = plan["S"] * G
    if path == "sweep":                                   # reduce_segments
        return rows if rows <= 16 else _cdiv(rows, 8) + 8
    if path == "tail":                                    # fused tail of the "obs" mapping
        ns = OBS_NT // plan["R"]
        return _cdiv(rows, ns) + ns
    return plan["S"] + G                                  # grad_finalize_chain / _coop


def planner_tags(plan, lens, tile=None):
    """The planner cases one plan takes (lens: group lengths)."""
    segs = [L for n in lens for L in segments(n, plan["S"])]
    tile = tile or (CH_TILE if plan["kind"] == "chains" else OBS_TILE)
    t = set()
    if plan["S"] == 1:
        t.add("S1")
    if plan.get("target", 0) > plan.get("max_S", 1 << 62):
        t.add("clamp")
    if plan.get("clamped", plan["S"]) != plan["S"]:
        t.add("cost")
    tr = plan.get("trace", [])
    if tr and tr[0] == (8, False, True) and plan["R"] < 8:
        t.add("fits")
    if plan["kind"] == "chains" and "R" in plan and plan["groups"] > 1 and plan.get("C", 0) % (CH_NT * plan["R"]):
        t.add("ragged")
    if any(L == 0 for L in segs):
        t.add("empty")
    if any(L > tile and L % tile for L in segs):
        t.add("fullpartial")
    if any(L % tile == 1 and L > tile for L in segs):
        t.add("tile+1")
    if any(L % tile == tile - 1 for L in segs):
        t.add("tile-1")
    if any(L % 2 for L in segs):
        t.add("oddtail")
    return t


def _plan_of(spec, sms):
    if spec["law"] == "mv":
        p = plan_gsnmv(spec["d"], spec["C"], spec["lens"][0], spec["force"], sms)
    else:
        p = plan_gsn1d(spec["C"], max(spec["lens"]), spec["force"], sms, len(spec["lens"]))
    p["C"] = spec["C"]
    return p


def _seg_len_shape(C, L, force, sms, G=1, d=None):
    """n such that the planner cuts segments of exactly L observations and a last one of L - 1 (L even,
    >= 256, so that max_S does not clamp): the plan's S is a fixed point of n = L S - 1."""
    S = (plan_gsnmv(d, C, 1 << 40, force, sms) if d else plan_gsn1d(C, 1 << 40, force, sms, G))["S"]
    for _ in range(8):
        n = L * S - 1
        S2 = (plan_gsnmv(d, C, n, force, sms) if d else plan_gsn1d(C, n, force, sms, G))["S"]
        if S2 == S:
            return n
        S = S2
    raise AssertionError(f"no fixed point for C={C} L={L} on {sms} SMs")


# ---- the cases ------------------------------------------------------------------------------------------

def _iid(C, n, force=0):
    return lambda sms: dict(law="iid", C=C, lens=[n], force=force)


def _iid_seg(C, L, force=0):
    return lambda sms: dict(law="iid", C=C, lens=[_seg_len_shape(C, L, force, sms)], force=force)


def _search(Cs, ns, tags, force=0):
    """The first (C, n) whose plan on `sms` SMs takes every case in `tags`."""
    def shape(sms):
        for C in Cs:
            for n in ns:
                spec = dict(law="iid", C=C, lens=[n], force=force)
                if set(tags) <= planner_tags(_plan_of(spec, sms), [n]):
                    return spec
        raise AssertionError(f"no shape takes {tags} on {sms} SMs")
    return shape


def _hier(C, lens, force=0):
    return lambda sms: dict(law="hier", C=C, lens=list(lens), force=force)


def _ragged_lens(G, seed, lo, hi):
    rng = np.random.default_rng(seed)
    lens = rng.integers(lo, hi, G)
    lens[:: max(1, G // 3)] |= 1                      # odd lengths
    if G >= 4:
        lens[1], lens[2] = 0, 1                       # an empty group and a single observation
    return [int(v) for v in lens]


def _mv(d, C, mapping, force=0):
    def shape(sms):
        p = plan_gsnmv(d, C, 1 << 40, force, sms)
        tile = p["tile"]
        m = _cdiv(256, tile)
        # chains: segments of m tiles + 2, the last one m tiles + 1; obs: m full tiles, the last one
        # a tile short of that (so cnt d is odd in the last tile whenever d is odd)
        L = m * tile + 2 if mapping == "chains" else max(m, 2) * tile
        return dict(law="mv", d=d, C=C, lens=[_seg_len_shape(C, L, force, sms, d=d)], force=force)
    return shape


# (name, shape of the SM count, regime, planner tags, expected variant).  Regimes (1-D): a = cfg 2-like
# (x ~ N(1.5, 2^2), mu near the mean); b = x = 1e6 + N(0, 1), mu near 1e6; c = mu 1e3 .. 1e8 away;
# d = mixed scales 10^+-3, exact zeros and a few |x| ~ 1e100; v1 / v2 = regime a with s2 ~ 1e-200 /
# 1e200; m = mu equal to the sample mean (T cancels); s = regime a with one (mu, s2) in every r-slot of
# a thread tile / every lane of an obs CTA.  gsnmv: a = well conditioned with a perturbed (unread)
# lower triangle, k = cond(Sigma) ~ 1e8, n = NaN in the lower triangle.
GSN1D_CASES = [
    ("r8_clamp", _search([4133, 4500], [30001, 20001, 10001], ["clamp", "ragged"]), "a", ["clamp", "ragged"], "gsn1d_chains_R8"),
    ("r8_tile+1", _iid_seg(2048, CH_TILE + 2), "b", ["tile+1", "oddtail"], "gsn1d_chains_R8"),
    ("r4_fits", _search([700, 600, 900], [100001, 150001, 200001, 300001], ["fits", "clamp"]), "c", ["fits", "clamp", "ragged"], "gsn1d_chains_R4"),
    ("r2_auto", _iid(300, 50001), "d", ["clamp", "ragged"], "gsn1d_chains_R2"),
    ("r1_s1", _iid(300, 255), "m", ["S1"], "gsn1d_chains_R1"),
    ("r1_auto", _iid(100, 20001), "v1", [], "gsn1d_chains_R1"),
    ("r1_tile-1", _iid_seg(200, CH_TILE, 11), "a", ["tile-1", "oddtail"], "gsn1d_chains_R1"),
    ("r2_cost", _search(range(513, 2304, 7), [120001], ["cost", "ragged"], 12), "a", ["cost", "ragged"], "gsn1d_chains_R2"),
    ("f11_c20", _iid(20, 3001, 11), "v2", [], "gsn1d_chains_R1"),
    ("f18_c5", _iid(5, 5000, 18), "d", [], "gsn1d_chains_R8"),
    ("f11_c127", _iid(127, 4097, 11), "b", [], "gsn1d_chains_R1"),
    ("f11_c129", _iid(129, 4099, 11), "a", [], "gsn1d_chains_R1"),
    ("f12_c255", _iid(255, 6001, 12), "c", [], "gsn1d_chains_R2"),
    ("f12_c257", _iid(257, 6003, 12), "m", [], "gsn1d_chains_R2"),
    ("f14_c511", _iid(511, 8001, 14), "a", [], "gsn1d_chains_R4"),
    ("f14_c513", _iid(513, 8003, 14), "d", [], "gsn1d_chains_R4"),
    ("f18_c1023", _iid(1023, 10001, 18), "s", [], "gsn1d_chains_R8"),
    ("f18_c1025", _iid(1025, 10003, 18), "v1", [], "gsn1d_chains_R8"),
    ("cb1_fullpartial", _iid_seg(1, OBS_TILE + 2), "a", ["fullpartial", "tile+1", "oddtail"], "gsn1d_obs_C1"),
    ("cb2_s1", _iid(2, 5), "m", ["S1", "oddtail"], "gsn1d_obs_C2"),
    ("cb4_c3", _iid(3, 700001), "b", ["clamp"], "gsn1d_obs_C4"),
    ("cb8_tile-1", _iid_seg(8, 2 * OBS_TILE), "c", ["fullpartial", "tile-1", "oddtail"], "gsn1d_obs_C8"),
    ("cb16_c9", _iid(9, 100001), "d", ["clamp"], "gsn1d_obs_C16"),
    ("cb32_c17", _iid(17, 50001), "v2", [], "gsn1d_obs_C32"),
    ("cb32_slots", _iid(32, 20001, 2), "s", [], "gsn1d_obs_C32"),
    ("cb32_v1", _iid(30, 9001), "v1", [], "gsn1d_obs_C32"),
    ("h1_chains", _hier(300, [5001]), "a", [], None),
    ("h2_obs", _hier(7, [1, 4001]), "a", ["empty", "oddtail"], "gsn1d_obs_C8"),
    ("h16_chains", _hier(513, _ragged_lens(16, 1, 40, 3000)), "a", ["empty", "oddtail"], None),
    ("h16_obs", _hier(20, _ragged_lens(16, 2, 500, 5000)), "b", ["empty"], "gsn1d_obs_C32"),
    ("h17_obs", _hier(32, _ragged_lens(17, 3, 100, 3000)), "c", ["empty"], "gsn1d_obs_C32"),
    ("h17_chains", _hier(200, _ragged_lens(17, 4, 100, 3000)), "d", ["empty"], None),
    ("h64_chains", _hier(1000, _ragged_lens(64, 5, 0, 2000)), "a", ["empty"], None),
    ("h64_obs", _hier(5, _ragged_lens(64, 6, 0, 1500)), "b", ["empty"], "gsn1d_obs_C8"),
]
MV_CASES = [(f"mv{d}_{m}", _mv(d, C, m, f), reg, tags, f"gsnmv_{m}")
            for d, C, m, f, reg, tags in [
                (2, 129, "chains", 0, "a", []), (2, 1, "obs", 0, "a", []),
                (3, 127, "chains", 0, "a", ["tile+1", "oddtail"]), (3, 7, "obs", 0, "a", ["tile-1", "oddtail"]),
                (4, 129, "chains", 0, "k", []), (4, 32, "obs", 0, "a", []),
                (5, 127, "chains", 0, "a", ["tile+1"]), (5, 40, "obs", 2, "a", ["tile-1"]),
                (6, 129, "chains", 0, "a", []), (6, 3, "obs", 0, "n", []),
                (7, 127, "chains", 0, "n", ["tile+1"]), (7, 16, "obs", 0, "a", ["tile-1"]),
                (8, 129, "chains", 0, "a", []), (8, 31, "obs", 0, "k", []),
                (9, 63, "chains", 0, "a", ["tile+1"]), (9, 5, "obs", 0, "a", ["tile-1"]),
                (10, 65, "chains", 0, "a", []), (10, 2, "obs", 0, "a", []),
                (11, 63, "chains", 0, "k", ["tile+1"]), (11, 9, "obs", 0, "a", ["tile-1"]),
                (12, 65, "chains", 0, "n", []), (12, 12, "obs", 0, "a", []),
                (13, 63, "chains", 0, "a", ["tile+1"]), (13, 1, "obs", 0, "k", ["tile-1"]),
                (14, 65, "chains", 0, "a", []), (14, 20, "obs", 0, "a", []),
                (15, 63, "chains", 0, "a", ["tile+1"]), (15, 25, "obs", 0, "n", ["tile-1"]),
                (16, 65, "chains", 0, "a", []), (16, 32, "obs", 0, "a", []),
            ]]
CASES = GSN1D_CASES + MV_CASES
CASE = {c[0]: c for c in CASES}


@functools.lru_cache(maxsize=None)
def case_spec(name, sms):
    _, shape, regime, tags, variant = CASE[name]
    spec = dict(shape(sms))
    spec.update(name=name, regime=regime, tags=tags, variant=variant)
    spec["plan"] = _plan_of(spec, sms)
    spec["taken"] = planner_tags(spec["plan"], spec["lens"], spec["plan"].get("tile"))
    return spec


def check_plan(name, sms):
    """The planner cases a case is meant to take, on `sms` SMs."""
    spec = case_spec(name, sms)
    p = spec["plan"]
    for t in spec["tags"]:
        assert t in spec["taken"], (name, sms, t, sorted(spec["taken"]), {k: v for k, v in p.items() if k != "trace"})
    if spec["variant"]:
        assert p["name"] == spec["variant"], (name, sms, p["name"])
    if name.startswith("h") and spec["variant"] is None:
        assert p["kind"] == "chains", (name, p["name"])
    return p


# ---- data ---------------------------------------------------------------------------------------------------

def _regime_1d(rng, regime, x, C):
    """Per-chain (mu, s2) of the 1-D regimes for data x."""
    xm, xv = float(np.mean(x)), float(np.var(x)) if x.size > 1 else 1.0
    if regime in ("a", "s", "v1", "v2"):
        mu = xm + 0.05 * rng.standard_normal(C)
        s2 = max(xv, 1e-3) * np.exp(0.1 * rng.standard_normal(C))
        if regime == "v1":
            s2 = 1e-200 * np.exp(0.1 * rng.standard_normal(C))
        elif regime == "v2":
            s2 = 1e200 * np.exp(0.1 * rng.standard_normal(C))
    elif regime == "b":
        mu = 1e6 + 0.05 * rng.standard_normal(C)
        s2 = np.exp(0.1 * rng.standard_normal(C))
    elif regime == "c":
        mu = xm + rng.choice([-1.0, 1.0], C) * 10.0 ** rng.uniform(3, 8, C)
        s2 = 10.0 ** rng.uniform(0, 10, C)
    elif regime == "d":
        mu = rng.standard_normal(C) * 10.0 ** rng.uniform(-3, 3, C)
        mu[::5] = rng.choice([-1.0, 1.0], mu[::5].size) * 1e99
        s2 = 10.0 ** rng.uniform(-3, 3, C)
    elif regime == "m":
        mu = np.full(C, xm)
        s2 = max(xv, 1e-3) * np.exp(0.1 * rng.standard_normal(C))
    else:
        raise AssertionError(regime)
    return mu, s2


def _data_1d(rng, regime, n):
    if regime == "b":
        return 1e6 + rng.standard_normal(n)
    if regime == "d":
        x = rng.standard_normal(n) * 10.0 ** rng.uniform(-3, 3, n)
        x[::97] = 0.0
        k = rng.choice(n, min(3, n), replace=False)
        x[k] = rng.choice([-1.0, 1.0], k.size) * rng.uniform(1, 2, k.size) * 1e100
        return x
    return 1.5 + 2.0 * rng.standard_normal(n)


def _slots(spec):
    """Chains that carry chain `first`'s parameters: every r-slot of one thread of a chains tile, or
    every lane of an obs CTA."""
    p = spec["plan"]
    if p["kind"] == "obs":
        return list(range(spec["C"]))
    return [5 + CH_NT * r for r in range(p["R"]) if 5 + CH_NT * r < spec["C"]]


@functools.lru_cache(maxsize=None)
def case_data(name, sms):
    """Observations, group lengths and the state [p][C] of a case."""
    spec = case_spec(name, sms)
    rng = np.random.default_rng(1000 + list(CASE).index(name))
    C, lens, regime = spec["C"], spec["lens"], spec["regime"]
    if spec["law"] == "iid":
        x = _data_1d(rng, regime, lens[0])
        mu, s2 = _regime_1d(rng, regime, x, C)
        th = np.vstack([mu, s2])
        if regime == "s":
            sl = _slots(spec)
            th[:, sl] = th[:, sl[:1]]
        return x, th
    if spec["law"] == "hier":
        G = len(lens)
        tg = 1.5 + 2.0 * rng.standard_normal(G)
        xs, th = [], np.empty((G + 2, C))
        for g, n in enumerate(lens):
            if regime == "d":
                xg = _data_1d(rng, "d", n)
            else:
                xg = tg[g] + rng.standard_normal(n) + (1e6 if regime == "b" else 0.0)
            xs.append(xg)
            m = float(np.mean(xg)) if n else tg[g]
            th[g] = m + 0.05 * rng.standard_normal(C)
            if regime == "c":
                th[g] += rng.choice([-1.0, 1.0], C) * 10.0 ** rng.uniform(3, 8, C)
            elif regime == "d":
                th[g] = rng.standard_normal(C) * 10.0 ** rng.uniform(-3, 3, C)
        th[G] = th[:G].mean(axis=0) + 0.1 * rng.standard_normal(C)
        th[G + 1] = np.exp(0.3 * rng.standard_normal(C))
        return np.concatenate(xs), th
    d, n = spec["d"], lens[0]
    Q, _ = np.linalg.qr(rng.standard_normal((d, d)))
    ev = np.logspace(0, -8, d) if regime == "k" else rng.uniform(0.5, 2.0, d)
    Sig0 = (Q * ev) @ Q.T
    Sig0 = (Sig0 + Sig0.T) / 2
    mu0 = rng.standard_normal(d)
    X = mu0 + rng.standard_normal((n, d)) @ np.linalg.cholesky(Sig0).T
    th = np.empty((d + d * d, C))
    th[:d] = mu0[:, None] + 0.05 * rng.standard_normal((d, C))
    scale = np.exp(0.1 * rng.standard_normal(C))
    for c in range(C):
        B = Sig0 * scale[c]
        if regime == "a":                  # a lower triangle that differs from the upper one (unread)
            low = np.tril(np.ones((d, d)), -1).astype(bool)
            B = B.copy()
            B[low] *= 1.0 + 0.2 * rng.standard_normal(low.sum())
        elif regime == "n":
            B = B.copy()
            B[np.tril(np.ones((d, d)), -1).astype(bool)] = np.nan
        th[d:, c] = B.T.ravel()            # vec(Sigma), column-major: B[r, col] at d + r + col d
    return X, th


# ---- references and bounds --------------------------------------------------------------------------------

def _group_stats(x):
    """m, A1, A2, sum |x - m| and n of one group (np.longdouble)."""
    n = x.size
    if n == 0:
        z = LD(0)
        return z, z, z, z, 0
    xl = x.astype(LD)
    m = xl.sum() / n
    e = xl - m
    return m, e.sum(), (e * e).sum(), np.abs(e).sum(), n


def _ref_err(n):
    return (40 + math.log2(max(n, 1))) * V64


def _sums(x, mu):
    """Per chain: S, T, M2, M1 and the reference's own error of S and T."""
    m, A1, A2, Aa, n = _group_stats(x)
    dl = m - mu.astype(LD)
    S = A2 + 2 * dl * A1 + n * dl * dl
    T = A1 + n * dl
    M2 = A2 + 2 * np.abs(dl * A1) + n * dl * dl
    M1 = Aa + n * np.abs(dl)
    return S, T, M2, M1, _ref_err(n) * M2, _ref_err(n) * M1


def gsn1d_depth(plan, lens, path, G=1):
    return max(thread_chain(plan, L) for n in lens for L in segments(n, plan["S"])) + reduce_depth(plan, path, G)


def iid_reference(x, th, plan, path):
    """ll, grad [2][C] (np.longdouble) and their bounds for GsnTargetLaw([0.0])."""
    mu, s2 = th[0], th[1].astype(LD)
    N = x.size
    S, T, M2, M1, eS, eT = _sums(x, mu)
    k = gsn1d_depth(plan, [N], path)
    dS = SAFETY * (k + 3) * U53 * M2 + eS
    dT = SAFETY * (k + 1) * U53 * M1 + eT
    lnv = np.log(s2)
    c0 = -(LOG2PI + lnv) / 2
    ll = N * c0 - S / (2 * s2)
    dc0 = 4 * U53 * (1 + LOG2PI / 2 + np.abs(lnv) / 2)
    b_ll = SAFETY * (N * dc0 + 2 * U53 * N * np.abs(c0) + (dS + 3 * U53 * S) / (2 * s2))
    g = np.vstack([T / s2, -N / (2 * s2) + S / (2 * s2 * s2)])
    b_g = SAFETY * np.vstack([(dT + U53 * np.abs(T)) / s2,
                              2 * U53 * N / (2 * s2) + (dS + 4 * U53 * S) / (2 * s2 * s2)])
    return dict(ll=ll, g=g, b_ll=b_ll, b_g=b_g, S=S, T=T, bS=dS, bT=dT)


def hier_reference(x, lens, th, plan, path):
    """ll, grad [G + 2][C] and their bounds for HierNormalLaw(G)."""
    G = len(lens)
    C = th.shape[1]
    N = sum(lens)
    mu, tau = th[G].astype(LD), th[G + 1].astype(LD)
    k = gsn1d_depth(plan, lens, path, G)
    S, M2s, eSs = np.zeros(C, LD), np.zeros(C, LD), np.zeros(C, LD)
    g, b_g = np.empty((G + 2, C), LD), np.empty((G + 2, C), LD)
    it2 = 1 / (tau * tau)
    dvs = th[:G].astype(LD) - mu
    off = 0
    for gi, n in enumerate(lens):
        Sg, Tg, M2, M1, eS, eT = _sums(x[off:off + n], th[gi])
        off += n
        S += Sg
        M2s += M2
        eSs += eS
        dT = SAFETY * (k + 1) * U53 * M1 + eT
        g[gi] = Tg - dvs[gi] * it2
        b_g[gi] = SAFETY * (dT + U53 * np.abs(Tg) + 6 * U53 * np.abs(dvs[gi]) * it2)
    D2 = (dvs * dvs).sum(axis=0)
    g[G] = dvs.sum(axis=0) * it2
    b_g[G] = SAFETY * (G + 4) * U53 * np.abs(dvs).sum(axis=0) * it2
    g[G + 1] = -G / tau + D2 * it2 / tau
    b_g[G + 1] = SAFETY * (2 * U53 * G / tau + (G + 6) * U53 * D2 * it2 / tau)
    dS = SAFETY * (k + 3) * U53 * M2s + eSs
    ll = -N * LOG2PI / 2 - S / 2 + G * (-LOG2PI / 2 - np.log(tau)) - D2 * it2 / 2
    mag = N * LOG2PI / 2 + S / 2 + G * (1 + np.abs(np.log(tau))) + D2 * it2 / 2
    b_ll = SAFETY * (dS / 2 + (G + 10) * U53 * mag)
    return dict(ll=ll, g=g, b_ll=b_ll, b_g=b_g, S=S, bS=dS)


def _sigma_blocks(th, d, upper=True):
    """Symmetric(triu(B)) (or, for the perturbation checks, Symmetric(tril(B))) per chain, [C][d][d]."""
    B = th[d:].T.reshape(-1, d, d).transpose(0, 2, 1).astype(LD)       # B[c, r, col]
    tri = np.triu(np.ones((d, d), bool)) if upper else np.tril(np.ones((d, d), bool))
    A = np.where(tri, B, LD(0))
    return A + np.where(np.eye(d, dtype=bool), LD(0), A.transpose(0, 2, 1))


def chol_ld(Sig):
    C, d, _ = Sig.shape
    L = np.zeros_like(Sig)
    for j in range(d):
        L[:, j, j] = np.sqrt(Sig[:, j, j] - (L[:, j, :j] ** 2).sum(axis=1))
        for i in range(j + 1, d):
            L[:, i, j] = (Sig[:, i, j] - (L[:, i, :j] * L[:, j, :j]).sum(axis=1)) / L[:, j, j]
    return L


def tri_inv_ld(L):
    C, d, _ = L.shape
    W = np.zeros_like(L)
    for j in range(d):
        W[:, j, j] = 1 / L[:, j, j]
        for i in range(j + 1, d):
            W[:, i, j] = -(L[:, i, j:i] * W[:, j:i, j]).sum(axis=1) / L[:, i, i]
    return W


def _gamma(n):
    return n * U53 / (1 - n * U53)


def mv_stats(X):
    n, d = X.shape
    Xl = X.astype(LD)
    m = Xl.sum(axis=0) / n
    E = Xl - m
    return m, E.sum(axis=0), E.T @ E, n


def mv_quad(W, M):
    """tr(W M W') per chain."""
    return np.einsum("cij,cjk,cik->c", W, M, W)


def mv_reference(X, th, plan, upper=True, transpose_w=False):
    """ll [C], its bound, S and its bound for sweep_gsnmv (W' / the lower triangle: perturbation checks)."""
    n, d = X.shape
    m, A1, A2, _ = mv_stats(X)
    dl = (m[:, None] - th[:d].astype(LD)).T                           # [C][d]
    M = A2[None] + A1[None, :, None] * dl[:, None, :] + dl[:, :, None] * A1[None, None, :] + \
        n * dl[:, :, None] * dl[:, None, :]
    L = chol_ld(_sigma_blocks(th, d, upper))
    W = tri_inv_ld(L)
    S = mv_quad(W.transpose(0, 2, 1) if transpose_w else W, M)
    logdet = np.log(np.diagonal(L, axis1=1, axis2=2)).sum(axis=1)
    c0 = -(d * LOG2PI + 2 * logdet) / 2
    ll = n * c0 - S / 2
    Wf, Lf = W.astype(np.float64), L.astype(np.float64)
    K = np.array([np.linalg.norm(np.abs(Wf[c]) @ np.abs(Lf[c]), 2) for c in range(Wf.shape[0])])
    eps_q = (_gamma(d + 1) + 2 * _gamma(d)) * K * K + 2 * (_gamma(d) + U53) * K + (d + 1) * U53
    k = max(thread_chain(plan, L_) for L_ in segments(n, plan["S"])) + reduce_depth(plan, "sweep")
    trM = np.trace(A2) + 2 * np.sqrt((A1 * A1).sum() * (dl * dl).sum(axis=1)) + n * (dl * dl).sum(axis=1)
    e_ref = (n + 8 * d + 40) * V64 * (W * W).sum(axis=(1, 2)) * trM
    bS = SAFETY * (eps_q + (k + 1) * U53) * S + e_ref
    ldabs = np.abs(np.log(np.diagonal(L, axis1=1, axis2=2))).sum(axis=1)
    dc0 = _gamma(d + 1) * d * K * K / 2 + (2 * d + 4) * U53 * (1 + d + ldabs)
    b_ll = SAFETY * (n * dc0 + 2 * U53 * n * np.abs(c0) + bS / 2 + U53 * S / 2)
    return dict(ll=ll, b_ll=b_ll, S=S, bS=bS, K=K)


def reference(name, sms, path, theta=None):
    spec = case_spec(name, sms)
    x, th = case_data(name, sms)
    th = th if theta is None else theta
    if spec["law"] == "iid":
        return iid_reference(x, th, spec["plan"], path)
    if spec["law"] == "hier":
        return hier_reference(x, spec["lens"], th, spec["plan"], path)
    return mv_reference(x, th, spec["plan"])


def within(part, got, ref, bound, where):
    """got (float64) against ref (longdouble) inside bound; where ref leaves the double range, the kernel
    returns the infinity of the same sign.  Returns the largest error / bound."""
    got = np.asarray(got, np.float64)
    with np.errstate(over="ignore"):
        refd = ref.astype(np.float64)
    over = np.isinf(refd)
    assert np.array_equal(got[over], refd[over]), (where, part, "overflow", got[over][:4], refd[over][:4])
    ok = ~over
    assert np.all(np.isfinite(got[ok])), (where, part, "not finite")
    err = np.abs(got[ok].astype(LD) - ref[ok])
    b = bound[ok]
    assert np.all(err[b == 0] == 0), (where, part, "exact zero expected")
    r = (err / np.where(b > 0, b, 1)).astype(np.float64)
    r[b == 0] = 0.0
    worst = float(r.max()) if r.size else 0.0
    idx = np.unravel_index(int(np.argmax(r)), r.shape) if r.size else None
    assert worst <= 1.0, (where, part, idx, worst)
    _note(part, worst)
    return worst


# ---- device runs ----------------------------------------------------------------------------------------------

def _ups():
    # the sessions only evaluate: any update will do
    return [em.RandomWalkUpdate(em.UniformRandomWalk([0.01]), [1])]


def _law(spec):
    if spec["law"] == "iid":
        return em.GsnTargetLaw([0.0]), None
    if spec["law"] == "hier":
        lens = spec["lens"]
        return em.HierNormalLaw(len(lens)), np.repeat(np.arange(len(lens)), lens).astype(np.float64)
    return em.GsnTargetLaw(np.zeros(spec["d"])), None


def run_case(name, sms, grad=True, env=None):
    """One session: variant, eval_loglik and (1-D laws) eval_grad."""
    spec = case_spec(name, sms)
    x, th = case_data(name, sms)
    law, y = _law(spec)
    # the library reads EXTMCMC_TAIL when it plans, at the first evaluation
    saved = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    g = None
    try:
        g = GpuSession(law, _ups(), x, th, spec["C"], y=y, sweep_variant=spec["force"])
        out = dict(variant=g.variant(), ll_loglik=g.eval_loglik(), launches=g.lib.extmcmc_launch_count(g.h))
        if grad and spec["law"] != "mv":
            out["ll_grad"], out["grad"] = g.eval_grad()
        assert g.lib.extmcmc_sync(g.h) == _abi.OK
    finally:
        if g is not None:
            g.close()
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return out


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def sms():
    return _sms()


def _inst(spec, grad):
    p = spec["plan"]
    if spec["law"] == "mv":
        return ("gsnmv", spec["d"], p["kind"])
    if spec["law"] == "hier":
        return ("hier", p["kind"], grad)
    return ("gsn1d", p["kind"], p["R"], grad)


_cases_done = set()


def check_gsn1d(name, sms, res, tail=True):
    spec = case_spec(name, sms)
    p = check_plan(name, sms)
    assert res["variant"] == p["name"], (name, res["variant"], p["name"])
    x, th = case_data(name, sms)
    tail_on = tail and spec["law"] == "iid" and p["kind"] == "obs"
    rv = reference(name, sms, "tail" if tail_on else "sweep")
    rg = reference(name, sms, "grad")
    w1 = within("1-D ll (eval_loglik)" if spec["law"] == "iid" else "hier ll (eval_loglik)",
                res["ll_loglik"], rv["ll"], rv["b_ll"], name)
    w2 = within("1-D ll (eval_grad)" if spec["law"] == "iid" else "hier ll (eval_grad)",
                res["ll_grad"], rg["ll"], rg["b_ll"], name)
    w3 = within("1-D grad" if spec["law"] == "iid" else "hier grad", res["grad"], rg["g"], rg["b_g"], name)
    print(f"{name} {p['name']} S={p['S']} C={spec['C']} N={sum(spec['lens'])} G={len(spec['lens'])} "
          f"({spec['regime']}): ll err / bound {w1:.3g} (loglik) {w2:.3g} (grad path), grad {w3:.3g}")
    if spec["regime"] == "s":
        sl = _slots(spec)
        for k in ("ll_loglik", "ll_grad"):
            assert np.all(res[k][sl] == res[k][sl[0]]), (name, k, res[k][sl])
        assert np.all(res["grad"][:, sl] == res["grad"][:, sl[:1]]), name
    _checked.add(_inst(spec, False))
    _checked.add(_inst(spec, True))
    _cases_done.add(name)


@pytest.mark.parametrize("name", [c[0] for c in GSN1D_CASES])
def test_gsn1d_every_chain(name, sms):
    check_gsn1d(name, sms, run_case(name, sms))


@pytest.mark.parametrize("name", ["cb1_fullpartial", "cb8_tile-1", "cb32_v1"])
def test_gsn1d_fused_tail_against_separate_reduction(name, sms):
    """EXTMCMC_TAIL=0 (read per plan): the separate reduce_segments pass instead of the last CTA's
    fixed-order tail; both inside the bound, equal to the last bits only (different association)."""
    fused, sep = run_case(name, sms, grad=False), run_case(name, sms, grad=False, env={"EXTMCMC_TAIL": "0"})
    rt, rs = reference(name, sms, "tail"), reference(name, sms, "sweep")
    w_t = within("1-D ll fused tail", fused["ll_loglik"], rt["ll"], rt["b_ll"], name)
    w_s = within("1-D ll separate reduction", sep["ll_loglik"], rs["ll"], rs["b_ll"], name)
    # the separate pass is one launch more (reduce_partials between the sweep and the finish)
    assert sep["launches"] == fused["launches"] + 1, (fused["launches"], sep["launches"])
    same = bool(np.array_equal(fused["ll_loglik"], sep["ll_loglik"]))
    print(f"{name}: fused tail err / bound {w_t:.3g}, separate {w_s:.3g}, bit-identical {same}")


@pytest.mark.parametrize("name", [c[0] for c in MV_CASES])
def test_gsnmv_every_chain(name, sms):
    spec = case_spec(name, sms)
    p = check_plan(name, sms)
    res = run_case(name, sms, grad=False)
    assert res["variant"] == p["name"], (name, res["variant"])
    r = reference(name, sms, "sweep")
    assert np.all(np.isfinite(res["ll_loglik"])), name          # NaN below the diagonal is never read
    w = within(f"gsnmv ll ({'cond 1e8' if spec['regime'] == 'k' else 'well conditioned'})",
               res["ll_loglik"], r["ll"], r["b_ll"], name)
    print(f"{name} d={spec['d']} S={p['S']} C={spec['C']} N={spec['lens'][0]} ({spec['regime']}): "
          f"ll err / bound {w:.3g}, K max {float(r['K'].max()):.3g}")
    _checked.add(_inst(spec, False))
    _cases_done.add(name)


# ---- the cooperative finish of the MALA kernels (G <= kCoopG = 16) against the per-chain one ---------------

@pytest.mark.parametrize("G", [16, 17])
def test_mala_step_finish_coop_and_chain(G, sms):
    """One replayed MALA step: mala_accept_kernel finishes the proposal's sums with grad_finalize_coop
    at G = 16 and grad_finalize_chain at G = 17 (mala_propose_kernel likewise for the current state)."""
    from oracle import oracle as orc
    lens = _ragged_lens(G, 40 + G, 50, 700)
    rng = np.random.default_rng(G)
    tg = 1.5 + 2.0 * rng.standard_normal(G)
    x = np.concatenate([tg[g] + rng.standard_normal(n) for g, n in enumerate(lens)])
    grp = np.repeat(np.arange(G), lens).astype(np.float64)
    C = 96
    th0 = np.empty((G + 2, C))
    th0[:G] = tg[:, None] + 0.05 * rng.standard_normal((G, C))
    th0[G], th0[G + 1] = tg.mean(), 1.5
    law = em.HierNormalLaw(G)
    ups = [em.MALAUpdate(0.02, list(range(1, G + 1)))]
    steps = list(em.MCMCSchedule(1, 1))
    ro = orc.Oracle(law, ups, x, th0, C, seed=G, y=grp).run(steps, n_threads=8)
    g = GpuSession(law, ups, x, th0, C, seed=G, n_steps_hint=4, y=grp)
    try:
        h = g.run(steps, replay=(ro["proposals"], ro["exp_draws"]))
        assert h["rc"] == _abi.OK
    finally:
        g.close()
    plan = plan_gsn1d(C, max(lens), 0, sms, G)
    w = []
    for th, ll, part in ((h["theta_prop"][0], h["ll_prop"][0], "proposal"), (h["theta"][0], h["ll"][0], "state")):
        r = hier_reference(x, lens, th, plan, "grad")
        w.append(within(f"MALA ll, G = {G} ({'coop' if G <= 16 else 'chain'} finish)", ll, r["ll"], r["b_ll"],
                        f"G={G} {part}"))
    print(f"MALA G={G}: ll err / bound {w[0]:.3g} (proposal), {w[1]:.3g} (state)")


# ---- the L2 evict_first copy at its real size ---------------------------------------------------------------

def l2_obs_count():
    import torch
    return 2 * (torch.cuda.get_device_properties(0).L2_cache_size // 16) + 4097


def run_l2(C, n):
    rng = np.random.default_rng(77 + C)
    x = 1.5 + 2.0 * rng.standard_normal(n)
    th = np.vstack([x.mean() + 0.05 * rng.standard_normal(C), 4.0 * np.exp(0.1 * rng.standard_normal(C))])
    g = GpuSession(em.GsnTargetLaw([0.0]), _ups(), x, th, C)
    try:
        out = dict(variant=np.array(g.variant()), ll_loglik=g.eval_loglik())
        out["ll_grad"], out["grad"] = g.eval_grad()
    finally:
        g.close()
    return x, th, out


_L2_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, %r)
from tests import test_gpu_gaussian_kernels as m
n, out = int(sys.argv[1]), sys.argv[2]
arrs = {}
for C in (8, 3):
    for k, v in m.run_l2(C, n)[2].items():
        arrs["%%d:%%s" %% (C, k)] = v
np.savez(out, **arrs)
print("done", len(arrs))
""" % ROOT


def test_l2_hint_path_at_its_real_size(sms, tmp_path):
    """Observations twice the size at which the bulk copies take the L2 evict_first policy (more than
    half of L2): cfg 5's shape C = 8 (CB = 8) and C = 3 (CB = 4), with and without the gradient; then
    the same in a process with EXTMCMC_L2_HINT=0 (read once per process): bit for bit."""
    n = l2_obs_count()
    res = {}
    for C in (8, 3):
        x, th, out = run_l2(C, n)
        plan = plan_gsn1d(C, n, 0, sms)
        assert str(out["variant"]) == plan["name"] == f"gsn1d_obs_C{8 if C == 8 else 4}"
        assert "fullpartial" in planner_tags(plan, [n]) or plan["S"] * OBS_TILE < n
        rv, rg = iid_reference(x, th, plan, "tail"), iid_reference(x, th, plan, "grad")
        w = (within("L2 hint: ll", out["ll_loglik"], rv["ll"], rv["b_ll"], f"L2 C={C}"),
             within("L2 hint: ll (grad path)", out["ll_grad"], rg["ll"], rg["b_ll"], f"L2 C={C}"),
             within("L2 hint: grad", out["grad"], rg["g"], rg["b_g"], f"L2 C={C}"))
        print(f"L2 path N={n} C={C} S={plan['S']}: err / bound {w[0]:.3g} {w[1]:.3g} {w[2]:.3g}")
        res[C] = out
    path = str(tmp_path / "l2off.npz")
    r = subprocess.run([sys.executable, "-c", _L2_CHILD, str(n), path], capture_output=True, text=True,
                       timeout=900, env=dict(os.environ, EXTMCMC_L2_HINT="0"), cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    z = np.load(path)
    for C, out in res.items():
        for k in ("ll_loglik", "ll_grad", "grad"):
            assert np.array_equal(z[f"{C}:{k}"], out[k]), (C, k)


def test_every_instantiation_was_checked():
    want = {("gsn1d", "chains", R, gr) for R in R_ALL for gr in (False, True)}
    want |= {("gsn1d", "obs", CB, gr) for CB in CB_ALL for gr in (False, True)}
    want |= {("hier", k, gr) for k in ("chains", "obs") for gr in (False, True)}
    want |= {("gsnmv", d, k) for d in range(2, 17) for k in ("chains", "obs")}
    if len(_cases_done) < len(CASES):
        pytest.skip("needs every case of the module in the same run")
    print("largest error / bound:", json.dumps(_worst, indent=1))
    assert want == _checked, sorted(want ^ _checked, key=str)
