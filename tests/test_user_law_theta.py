"""User-defined laws with a term of theta only, without a device (extmcmc_user_law_check_ex,
DeviceLaw(..., theta_term=True)): every sample law compiles without spills in every mode and chunk
width, a source lacking a function the flag declares is refused with a log that names it, the argument
checks of the _ex entry points, and the Python constructor."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws as ul
from tests import user_laws_theta as ut

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 10


def _check(src, P, D, with_grad, chunk=0, flags=_abi.USER_THETA_TERM):
    buf = C.create_string_buffer(1 << 20)
    used = C.c_int32(-1)
    rc = _abi.load().extmcmc_user_law_check_ex(src.encode(), P, D, with_grad, chunk, flags, C.byref(used), buf, len(buf))
    return rc, used.value, buf.value.decode()


def _kernels(log):
    """entry function -> (spill stores, spill loads, registers)"""
    return {m.group(1): (int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in re.finditer(
        r"Function properties for (extmcmc_user_\w+)\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads\n"
        r".*?Used (\d+) registers", log)}


def _rmax(n):
    return 4 if 4 * n <= 40 else 2 if 2 * n <= 40 else 1


# (name, with_grad, chunk): plain, hand-written, forward unchunked, and chunk widths 3 and 5 at P = 10
MODES = [(_abi.USER_GRAD_NONE, 0), (_abi.USER_GRAD_HAND, 0), (_abi.USER_GRAD_FORWARD, 0),
         (_abi.USER_GRAD_FORWARD, 3), (_abi.USER_GRAD_FORWARD, 5)]


@pytest.mark.parametrize("with_grad,chunk", MODES)
@pytest.mark.parametrize("name", list(ut.LAWS))
def test_every_instantiation_compiles_without_spills(name, with_grad, chunk):
    hand, fwd, Df, _, _ = ut.LAWS[name]
    src = fwd if with_grad == _abi.USER_GRAD_FORWARD else hand
    rc, used, log = _check(src, P, Df(P), with_grad, chunk)
    assert rc == _abi.OK, log
    ks = _kernels(log)
    if with_grad == _abi.USER_GRAD_FORWARD:
        K = chunk or P
        assert used == K
        nc = -(-P // K)
        rs = [r for r in (1, 2, 4) if r <= _rmax((P + 1) * (K + 1))]
        sfx = ["_f"] if nc == 1 else [f"_f{K}c{c}" for c in range(nc)]
        expect = {f"extmcmc_user_chains_r{r}{s}" for r in rs for s in sfx + ["_g0"]}
        expect |= {f"extmcmc_user_lanes{s}" for s in sfx + ["_g0"]}
    else:
        assert used == 0
        gs = ["_g0", "_g1"] if with_grad else ["_g0"]
        rs = [r for r in (1, 2, 4) if r <= _rmax(2 * P + 1 if with_grad else P + 1)]
        expect = {f"extmcmc_user_chains_r{r}{g}" for r in rs for g in gs} | {f"extmcmc_user_lanes{g}" for g in gs}
    assert set(ks) == expect, sorted(set(ks) ^ expect)
    assert all(v[:2] == (0, 0) for v in ks.values()), {k: v for k, v in ks.items() if v[:2] != (0, 0)}


@pytest.mark.parametrize("src,with_grad,missing", [
    (ut.NO_THETA_PLAIN, _abi.USER_GRAD_NONE, "logpdf_theta"),
    (ut.NO_THETA_PLAIN, _abi.USER_GRAD_HAND, "logpdf_theta"),
    (ut.NO_THETA_GRAD, _abi.USER_GRAD_HAND, "logpdf_theta_grad"),
    (ut.NO_THETA_FORWARD, _abi.USER_GRAD_FORWARD, "logpdf_theta")])
def test_a_declared_term_that_is_missing_does_not_compile(src, with_grad, missing):
    Pm = P if src is ut.NO_THETA_GRAD else 8
    D = 2 if src is ut.NO_THETA_GRAD else 8
    rc, used, log = _check(src, Pm, D, with_grad)
    assert rc == _abi.EINVAL, log
    assert re.search(r'identifier "%s" is undefined|"%s"' % (missing, missing), log), log
    assert used == (Pm if with_grad == _abi.USER_GRAD_FORWARD else 0)
    # without the flag the same source compiles: the term is declared, not detected
    if src is not ut.NO_THETA_GRAD:
        assert _check(src, Pm, D, with_grad, flags=0)[0] == _abi.OK


def test_argument_checks():
    for bad in (2, 3, -1, 1 << 30):
        rc, used, log = _check(ut.HIER, P, 2, _abi.USER_GRAD_NONE, flags=bad)
        assert rc == _abi.EINVAL and used == -1 and "flags" in log, (bad, log)
    for with_grad in (_abi.USER_GRAD_NONE, _abi.USER_GRAD_HAND):
        rc, used, log = _check(ut.HIER_HAND, P, 2, with_grad, chunk=2)
        assert rc == _abi.EINVAL and used == -1 and "chunk must be 0 unless" in log, log
    # chunk keeps the meaning of the _chunked entry points in forward mode
    rc, used, log = _check(ut.HIER_FORWARD, P, 2, _abi.USER_GRAD_FORWARD, chunk=11)
    assert rc == _abi.EINVAL and used == -1 and "chunk" in log
    rc, used, log = _check(ut.RIDGE_POISSON_FORWARD, 24, 23, _abi.USER_GRAD_FORWARD, chunk=0)
    assert (rc, used) == (_abi.OK, 5), log
    assert _check(ut.HIER, 65, 2, _abi.USER_GRAD_NONE)[0] == _abi.EUNSUPPORTED
    assert _abi.load().extmcmc_set_user_law_ex(None, ut.HIER.encode(), 0, 0, _abi.USER_THETA_TERM) == _abi.EINVAL


def test_without_flags_the_ex_entry_point_is_the_existing_program():
    # the same input as the existing entry points: the same cached result and log
    buf = C.create_string_buffer(1 << 20)
    rc0 = _abi.load().extmcmc_user_law_check(ul.POISSON_REG.encode(), 8, 8, _abi.USER_GRAD_HAND, buf, len(buf))
    rc, used, log = _check(ul.POISSON_REG, 8, 8, _abi.USER_GRAD_HAND, flags=0)
    assert (rc, used, log) == (rc0, 0, buf.value.decode())


def test_device_law_theta_term_argument():
    law = em.DeviceLaw(ut.HIER, P, 2, theta_term=True)
    assert law.theta_term is True and law.chunk is None and law.gradient is False
    assert em.DeviceLaw(ut.HIER, P, 2).theta_term is False
    assert em.DeviceLaw(ut.HIER_HAND, P, 2, gradient=True, theta_term=True).gradient is True
    assert em.DeviceLaw(ut.HIER_FORWARD, P, 2, gradient="forward", theta_term=True).chunk == P
    assert em.DeviceLaw(ut.HIER_FORWARD, P, 2, gradient="forward", chunk=3, theta_term=True).chunk == 3
    assert em.DeviceLaw(ut.RIDGE_POISSON_FORWARD, 24, 23, gradient="forward", chunk="auto", theta_term=True).chunk == 5
    for bad in (1, 0, None, "yes", 1.0):
        with pytest.raises(ValueError, match="theta_term must be True or False"):
            em.DeviceLaw(ut.HIER, P, 2, theta_term=bad)
    with pytest.raises(ValueError, match="does not compile"):
        em.DeviceLaw(ut.NO_THETA_GRAD, P, 2, gradient=True, theta_term=True)
    with pytest.raises(ValueError, match="chunk"):
        em.DeviceLaw(ut.HIER_FORWARD, P, 2, gradient="forward", chunk=11, theta_term=True)


def test_sass_fp64_counts_of_the_existing_laws_are_unchanged():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "user_law_sass_fp64.py")], capture_output=True,
                         text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    # the row loop is unrolled 4 times: its FP64 count is 4 x the count per chain x row
    loops = lambda block: {int(x) for x in re.findall(r"loop \S+ fp64 (\d+) of", block)}  # noqa: E731
    hand, fwd = out.stdout.split("forward kernel")
    assert 4 * 51 in loops(hand) and 4 * 115 in loops(fwd), out.stdout
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "user_law_sass_fp64.py"), "--chunked", "32", "5"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    chunks = out.stdout.split("forward chunk")[1:]
    assert len(chunks) == 7, out.stdout
    # per chunk: the one-row remainder loop beside the unrolled one
    assert sum(max(x for x in loops(b) if x and 4 * x in loops(b)) for b in chunks) == 1558, out.stdout
