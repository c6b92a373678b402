"""Host-only half of tests/test_gpu_gaussian_kernels.py: the planner mirror takes the intended case for
every shape on a B200's 148 SMs, and every derived bound discriminates -- on the data regime (a)
shapes, a reference that drops the last observation of the data or of a group, counts one zero padding
element, moves one observation to the neighbouring group, takes the neighbouring chain's T, or (gsnmv)
uses W' in place of W or the lower triangle of Sigma in place of the upper one falls outside the bound
of at least one output on every chain."""
import numpy as np
import pytest

from tests import test_gpu_gaussian_kernels as gk

LD = np.longdouble
SMS = 148
A_1D = [c[0] for c in gk.GSN1D_CASES if c[2] == "a"]
A_MV = [c[0] for c in gk.MV_CASES if c[2] == "a"]


@pytest.mark.parametrize("name", list(gk.CASE))
def test_planner_case_on_148_sms(name):
    gk.check_plan(name, SMS)


def test_every_instantiation_is_planned_on_148_sms():
    got = set()
    for name in gk.CASE:
        spec = gk.case_spec(name, SMS)
        got |= {gk._inst(spec, False), gk._inst(spec, True)} if spec["law"] != "mv" else {gk._inst(spec, False)}
    want = {("gsn1d", "chains", R, gr) for R in gk.R_ALL for gr in (False, True)}
    want |= {("gsn1d", "obs", CB, gr) for CB in gk.CB_ALL for gr in (False, True)}
    want |= {("hier", k, gr) for k in ("chains", "obs") for gr in (False, True)}
    want |= {("gsnmv", d, k) for d in range(2, 17) for k in ("chains", "obs")}
    assert got == want, sorted(got ^ want, key=str)


def test_planner_mirror_follows_chains_ctas(monkeypatch):
    base = gk.plan_gsn1d(4096, 1_000_000, 0, SMS)
    assert (base["R"], base["S"]) == (8, 296)                   # cfg 2: 4 groups x 296 = 8 CTAs per SM
    monkeypatch.setenv("EXTMCMC_CHAINS_CTAS", "4")
    assert gk.plan_gsn1d(4096, 1_000_000, 0, SMS)["S"] == 148
    monkeypatch.setenv("EXTMCMC_CHAINS_CTAS", "0")               # atoi <= 0: the default
    assert gk.plan_gsn1d(4096, 1_000_000, 0, SMS)["S"] == 296


@pytest.mark.parametrize("sms", [132, 160])
def test_searched_shapes_exist_for_other_sm_counts(sms):
    for name, shape, *_ in gk.CASES:
        spec = dict(shape(sms))
        taken = gk.planner_tags(gk._plan_of(spec, sms), spec["lens"], gk._plan_of(spec, sms).get("tile"))
        want = {t for t in gk.CASE[name][3] if t in ("fits", "cost", "tile+1", "tile-1")}
        assert want <= taken, (name, sms, want - taken)


def _outside_1d(ref, dS, dT, s2):
    """Per chain: does a reference whose S, T moved by dS, dT leave the bound of ll, d/dmu or d/ds2?"""
    s2 = s2.astype(LD)
    return ((np.abs(dS / (2 * s2)) > ref["b_ll"]) | (np.abs(dT / s2) > ref["b_g"][0]) |
            (np.abs(dS / (2 * s2 * s2)) > ref["b_g"][1]))


@pytest.mark.parametrize("name", [n for n in A_1D if gk.CASE[n][1](SMS)["law"] == "iid"])
def test_iid_bounds_discriminate(name):
    x, th = gk.case_data(name, SMS)
    mu = th[0].astype(LD)
    for path in ("sweep", "tail", "grad"):
        r = gk.reference(name, SMS, path)
        e = LD(x[-1]) - mu
        assert np.all(_outside_1d(r, -e * e, -e, th[1])), (name, path, "last observation dropped")
        assert np.all(_outside_1d(r, mu * mu, -mu, th[1])), (name, path, "zero padding element counted")
        T = r["T"]
        nb = np.roll(T, -1)
        assert T.size < 2 or np.all(np.abs((nb - T) / th[1].astype(LD)) > r["b_g"][0]), (name, path, "neighbouring chain's T")


def _group_T(x, lens, th):
    out, off = [], 0
    for g, n in enumerate(lens):
        out.append(gk._sums(x[off:off + n], th[g])[1])
        off += n
    return out


@pytest.mark.parametrize("name", [n for n in A_1D if gk.CASE[n][1](SMS)["law"] == "hier"])
def test_hier_bounds_discriminate(name):
    spec = gk.case_spec(name, SMS)
    lens = spec["lens"]
    x, th = gk.case_data(name, SMS)
    r = gk.reference(name, SMS, "grad")
    T = _group_T(x, lens, th)
    ends = np.cumsum(lens)
    for g, n in enumerate(lens):
        thg = th[g].astype(LD)
        assert np.all(np.abs(thg) > r["b_g"][g]), (name, g, "zero padding element counted")
        if n == 0:
            continue
        e = LD(x[ends[g] - 1]) - thg
        assert np.all(np.abs(e) > r["b_g"][g]), (name, g, "last observation of the group dropped")
        if g + 1 < len(lens):
            e2 = LD(x[ends[g] - 1]) - th[g + 1].astype(LD)
            assert np.all((np.abs(e) > r["b_g"][g]) | (np.abs(e2) > r["b_g"][g + 1])), (name, g, "moved")
        if g > 0 and lens[g - 1] > 0:
            e0 = LD(x[ends[g - 1]]) - thg                       # first of group g into group g - 1
            e1 = LD(x[ends[g - 1]]) - th[g - 1].astype(LD)
            assert np.all((np.abs(e0) > r["b_g"][g]) | (np.abs(e1) > r["b_g"][g - 1])), (name, g, "moved back")
        assert np.all(np.abs(np.roll(T[g], -1) - T[g]) > r["b_g"][g]), (name, g, "neighbouring chain's T")


@pytest.mark.parametrize("name", A_MV)
def test_gsnmv_bounds_discriminate(name):
    spec = gk.case_spec(name, SMS)
    x, th = gk.case_data(name, SMS)
    r = gk.mv_reference(x, th, spec["plan"])
    wt = gk.mv_reference(x, th, spec["plan"], transpose_w=True)
    lo = gk.mv_reference(x, th, spec["plan"], upper=False)
    assert np.all(np.abs(wt["S"] - r["S"]) > r["bS"]), (name, "W' in place of W")
    assert np.all(np.abs(lo["ll"] - r["ll"]) > r["b_ll"]), (name, "lower triangle in place of the upper one")
    # and the padding element of an odd tail, read as one more observation x = 0
    d = spec["d"]
    e = -th[:d].astype(LD)
    Lf = gk.chol_ld(gk._sigma_blocks(th, d))
    z = np.einsum("cij,jc->ci", gk.tri_inv_ld(Lf), e)
    assert np.all((z * z).sum(axis=1) > r["bS"]), (name, "zero padding observation counted")


def test_bounds_are_tight_enough_to_matter():
    """The relative size of the S bound on the cfg 2-like shapes: far below the effect of one
    observation in 1e5 (so a tile-edge off-by-one cannot hide in it)."""
    for name in A_1D[:3]:
        r = gk.reference(name, SMS, "grad")
        rel = (r["bS"] / r["S"]).astype(np.float64) if "bS" in r else None
        assert rel is not None and rel.max() < 1e-9, (name, rel.max())
