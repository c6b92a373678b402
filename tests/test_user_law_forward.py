"""Forward-mode gradients of user-defined laws without a device: the templated sample laws compile at
every instantiation the planner can pick with 0 spill bytes, what Dual cannot differentiate does not
compile, the parameter limit, the Python constructor, and csrc/dual.cuh itself, built as host code:
every overload's tangents against mpmath derivatives and its values against the plain double call."""
import ctypes as C
import os
import re
import shutil
import subprocess

import mpmath
import numpy as np
import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws_forward as uf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "extensiblemcmc.jl_b200", "csrc")


def _check(src, P, D, with_grad):
    buf = C.create_string_buffer(1 << 18)
    rc = _abi.load().extmcmc_user_law_check(src.encode(), P, D, with_grad, buf, len(buf))
    return rc, buf.value.decode()


def _rmax_forward(P):
    """user_max_R (sweep_user.cuh) in forward mode: (P + 1)^2 doubles per chain."""
    n = (P + 1) ** 2
    return 4 if 4 * n <= 40 else 2 if 2 * n <= 40 else 1


# the four laws at P <= 8 (the regression laws take P from D)
FWD_SHAPES = [("gsn1d", 2, 1), ("poisson_rate", 1, 1),
              ("logistic", 1, 2), ("logistic", 2, 3), ("logistic", 4, 5), ("logistic", 8, 9),
              ("poisson_reg", 1, 1), ("poisson_reg", 3, 3), ("poisson_reg", 5, 5), ("poisson_reg", 8, 8)]


@pytest.mark.parametrize("name,P,D", FWD_SHAPES)
def test_forward_laws_compile_without_spills(name, P, D):
    rc, log = _check(uf.LAWS[name][0], P, D, _abi.USER_GRAD_FORWARD)
    assert rc == _abi.OK, log
    blocks = re.findall(r"Compiling entry function '(extmcmc_user_\w+)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads",
                        log, re.S)
    spills = {k: (int(st), int(ld)) for k, st, ld in blocks}
    rmax = _rmax_forward(P)
    # value kernels on Law<double>, forward kernels on Law<Dual<P>>, under their own names
    expect = {f"extmcmc_user_chains_r{r}_{g}" for r in (1, 2, 4) if r <= rmax for g in ("g0", "f")}
    expect |= {"extmcmc_user_lanes_g0", "extmcmc_user_lanes_f"}
    assert set(spills) == expect, (sorted(spills), log)
    assert all(s == (0, 0) for s in spills.values()), spills
    assert "sm_100a" in log


def test_forward_mode_leaves_the_hand_gradient_kernels_alone():
    # with_grad = 1 still means logpdf_grad: the same kernel names as before, no forward kernels
    from tests import user_laws as ul
    rc, log = _check(ul.POISSON_REG, 3, 3, _abi.USER_GRAD_HAND)
    assert rc == _abi.OK, log
    assert "_g1" in log and "_f'" not in log and "Dual" not in log
    # any other non-zero with_grad is "hand-written" too
    assert _check(ul.POISSON_REG, 3, 3, 7) == (rc, log)


@pytest.mark.parametrize("src,needle", [(uf.BAD_LGAMMA, "lgamma"), (uf.BAD_NARROW, "const double lam = L.lam")])
def test_what_dual_cannot_differentiate_does_not_compile(src, needle):
    rc, log = _check(src, 1, 1, _abi.USER_GRAD_FORWARD)
    assert rc == _abi.EINVAL, log
    # the user's line, the call, and the dual instantiation it failed in
    assert re.search(r"law\(\d+\): error", log) and needle in log and "Dual<1>" in log, log


def test_forward_mode_parameter_limit():
    rc, log = _check(uf.POISSON_REG, 17, 17, _abi.USER_GRAD_FORWARD)
    assert rc == _abi.EUNSUPPORTED and "n_params <= 16" in log, log
    assert "n_params <= 16" in _abi.load().extmcmc_last_error(None).decode()
    with pytest.raises(_abi.ExtMCMCError) as ei:
        em.DeviceLaw(uf.POISSON_REG, 17, 17, gradient="forward")
    assert ei.value.code == _abi.EUNSUPPORTED
    # the hand-written contract keeps its own limit of 64
    from tests import user_laws as ul
    assert _check(ul.POISSON_REG, 17, 17, _abi.USER_GRAD_HAND)[0] == _abi.OK


def test_device_law_gradient_modes():
    law = em.DeviceLaw(uf.POISSON_REG, 3, 3, gradient="forward")
    assert (law.abi_law(), law.n_params, law.obs_dim, law.gradient) == (_abi.LAW_USER, 3, 3, "forward")
    assert "extmcmc_user_lanes_f" in law.log
    from tests import user_laws as ul
    assert em.DeviceLaw(ul.POISSON_RATE, 1, 1, gradient=False).gradient is False
    assert em.DeviceLaw(ul.POISSON_REG, 3, 3, gradient=True).gradient is True
    for bad in ("Forward", "hand", None, 2, 0.5, [True]):
        with pytest.raises(ValueError, match="gradient must be"):
            em.DeviceLaw(ul.POISSON_RATE, 1, 1, gradient=bad)
    # a templated source is a forward-mode law only
    for mode in (False, True):
        with pytest.raises(ValueError, match="does not compile"):
            em.DeviceLaw(uf.POISSON_RATE, 1, 1, gradient=mode)


def test_set_user_law_forward_needs_a_handle():
    assert _abi.load().extmcmc_set_user_law(None, uf.GSN1D.encode(), _abi.USER_GRAD_FORWARD) == _abi.EINVAL


# ---- dual.cuh as host code --------------------------------------------------------------------------

_HOST = r"""
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
static double normcdf(double x) { return 0.5 * erfc(-x * 0.70710678118654752); }
#include "dual.cuh"
using extmcmc::Dual;
typedef Dual<2> D2;
static D2 var(double v, int k) { D2 r(v); r.t[k] = 1.0; return r; }
static int bad = 0;
static void out(const char *name, double x, double y, const D2 &r, double plain) {
    uint64_t a, b;
    memcpy(&a, &r.v, 8); memcpy(&b, &plain, 8);
    if (a != b) { ++bad; fprintf(stderr, "value mismatch %s %a %a: %a vs %a\n", name, x, y, r.v, plain); }
    printf("%s %a %a %a %a %a\n", name, x, y, r.v, r.t[0], r.t[1]);
}
#define U(f, x) out(#f, x, 0.0, extmcmc::f(var(x, 0)), ::f(x))
int main() {
    const double all[] = {-2.5, -1.0, -0.3, 0.2, 0.7, 1.5, 3.0};
    const double pos[] = {0.1, 0.7, 1.5, 3.0, 10.0};
    const double gt1[] = {-0.5, -0.1, 0.3, 2.0, 40.0};
    for (double x : all) {
        U(exp, x); U(expm1, x); U(sin, x); U(cos, x); U(tanh, x); U(erf, x); U(erfc, x); U(normcdf, x);
        U(fabs, x);
        out("neg", x, 0.0, -var(x, 0), -x);
    }
    for (double x : pos) { U(log, x); U(sqrt, x); }
    for (double x : gt1) U(log1p, x);
    for (double x : all) for (double y : all) {
        const D2 a = var(x, 0), b = var(y, 1);
        out("add", x, y, a + b, x + y); out("sub", x, y, a - b, x - y);
        out("mul", x, y, a * b, x * y); out("div", x, y, a / b, x / y);
        out("add_dd", x, y, a + y, x + y); out("add_nd", x, y, x + b, x + y);
        out("sub_dd", x, y, a - y, x - y); out("sub_nd", x, y, x - b, x - y);
        out("mul_dd", x, y, a * y, x * y); out("mul_nd", x, y, x * b, x * y);
        out("div_dd", x, y, a / y, x / y); out("div_nd", x, y, x / b, x / y);
        D2 c = a; c += b; out("add", x, y, c, x + y);
        c = a; c -= b; out("sub", x, y, c, x - y);
        c = a; c *= b; out("mul", x, y, c, x * y);
        c = a; c /= b; out("div", x, y, c, x / y);
        c = a; c *= y; out("mul_dd", x, y, c, x * y);
        out("fmax", x, y, extmcmc::fmax(a, b), ::fmax(x, y)); out("fmin", x, y, extmcmc::fmin(a, b), ::fmin(x, y));
        out("fmax_dd", x, y, extmcmc::fmax(a, y), ::fmax(x, y)); out("fmin_nd", x, y, extmcmc::fmin(x, b), ::fmin(x, y));
        out("fma_ddn", x, y, extmcmc::fma(a, b, 0.25), ::fma(x, y, 0.25));
        out("fma_dnd", x, y, extmcmc::fma(a, 1.75, b), ::fma(x, 1.75, y));
        out("fma_ndd", x, y, extmcmc::fma(1.75, a, b), ::fma(1.75, x, y));
        const bool cmp = (a < b) == (x < y) && (a <= y) == (x <= y) && (x > b) == (x > y) && (a >= b) == (x >= y) &&
                         (a == b) == (x == y) && (a != y) == (x != y);
        if (!cmp) { ++bad; fprintf(stderr, "comparison %a %a\n", x, y); }
    }
    for (double x : pos) for (double y : all) {
        const D2 a = var(x, 0), b = var(y, 1);
        out("pow", x, y, extmcmc::pow(a, b), ::pow(x, y));
        out("pow_dd", x, y, extmcmc::pow(a, y), ::pow(x, y));
        out("pow_nd", x, y, extmcmc::pow(x, b), ::pow(x, y));
    }
    const double inf = 1.0 / 0.0, nan = 0.0 / 0.0;
    if (!extmcmc::isinf(D2(inf)) || extmcmc::isinf(D2(1.0)) || !extmcmc::isnan(D2(nan)) || extmcmc::isnan(D2(1.0)) ||
        extmcmc::isfinite(D2(inf)) || !extmcmc::isfinite(D2(1.0))) { ++bad; fprintf(stderr, "classification\n"); }
    // conventions: fabs at +-0 takes sign +1; fmax / fmin on a tie take the first operand's tangents
    out("fabs0", 0.0, 0.0, extmcmc::fabs(var(0.0, 0)), 0.0);
    out("fabs0", -0.0, 0.0, extmcmc::fabs(var(-0.0, 0)), 0.0);
    out("fmax_tie", 1.0, 1.0, extmcmc::fmax(var(1.0, 0), var(1.0, 1)), 1.0);
    out("fmin_tie", 1.0, 1.0, extmcmc::fmin(var(1.0, 0), var(1.0, 1)), 1.0);
    return bad;
}
"""


@pytest.fixture(scope="module")
def dual_table(tmp_path_factory):
    cxx = shutil.which("g++") or shutil.which("c++")
    if not cxx:
        pytest.skip("no host C++ compiler")
    d = tmp_path_factory.mktemp("dual")
    (d / "t.cpp").write_text(_HOST)
    exe = d / "t"
    # -ffp-contract=off: the library compiles its laws with -fmad=false
    subprocess.run([cxx, "-std=c++17", "-O2", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas",
                    "-I", CSRC, str(d / "t.cpp"), "-o", str(exe), "-lm"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr           # values equal the plain double call, bit for bit
    rows = []
    for line in r.stdout.splitlines():
        name, *vals = line.split()
        rows.append((name, *[float.fromhex(v) for v in vals]))
    return rows


mpmath.mp.dps = 40
_UNARY = {"exp": mpmath.exp, "expm1": mpmath.expm1, "sin": mpmath.sin, "cos": mpmath.cos, "tanh": mpmath.tanh,
          "erf": mpmath.erf, "erfc": mpmath.erfc, "normcdf": mpmath.ncdf, "log": mpmath.log, "sqrt": mpmath.sqrt,
          "log1p": mpmath.log1p, "neg": lambda x: -x}


def _partials(name, x, y):
    """(d/dx, d/dy) in 40 digits; for the _dd / _nd forms the double operand has no tangent."""
    x, y = mpmath.mpf(x), mpmath.mpf(y)
    base = name.split("_")[0].rstrip("0")
    if base in _UNARY:
        return mpmath.diff(_UNARY[base], x), 0
    if base == "fabs":
        return (-1 if x < 0 else 1), 0
    if base == "fma":      # operands: (dual x, dual y, 0.25), (dual x, 1.75, dual y), (1.75, dual x, dual y)
        return {"fma_ddn": (y, x), "fma_dnd": (1.75, 1), "fma_ndd": (1.75, 1)}[name]
    f = {"add": lambda a, b: a + b, "sub": lambda a, b: a - b, "mul": lambda a, b: a * b, "div": lambda a, b: a / b,
         "pow": lambda a, b: a ** b}.get(base)
    if base in ("fmax", "fmin"):
        first = x >= y if base == "fmax" else x <= y
        dx, dy = (1, 0) if first else (0, 1)
    else:
        dx = mpmath.diff(lambda a: f(a, y), x)
        dy = mpmath.diff(lambda b: f(x, b), y)
    if name.endswith("_dd"):
        dy = 0
    if name.endswith("_nd"):
        dx = 0
    return dx, dy


def test_dual_tangents_against_mpmath(dual_table):
    worst = 0.0
    names = set()
    for name, x, y, v, t0, t1 in dual_table:
        names.add(name.split("_")[0])
        for t, ref in zip((t0, t1), _partials(name, x, y)):
            ref = float(ref) if not isinstance(ref, float) else ref
            err = abs(t - ref)
            assert err <= 1e-14 * abs(ref), (name, x, y, t, ref)
            if ref:
                worst = max(worst, err / abs(ref))
    print(f"{len(dual_table)} cases, worst relative tangent error {worst:.3g}")
    assert names >= {"exp", "expm1", "log", "log1p", "sqrt", "pow", "fabs", "fmin", "fmax", "fma", "sin", "cos",
                     "tanh", "erf", "erfc", "normcdf", "add", "sub", "mul", "div", "neg"}


def test_dual_conventions(dual_table):
    conv = [(name, x, t0, t1) for name, x, y, v, t0, t1 in dual_table if name in ("fabs0", "fmax_tie", "fmin_tie")]
    assert [(n, np.copysign(1.0, x), t0, t1) for n, x, t0, t1 in conv] == [
        ("fabs0", 1.0, 1.0, 0.0), ("fabs0", -1.0, 1.0, 0.0),       # +0 and -0: sign +1
        ("fmax_tie", 1.0, 1.0, 0.0), ("fmin_tie", 1.0, 1.0, 0.0)]  # a tie: the first operand's tangents
