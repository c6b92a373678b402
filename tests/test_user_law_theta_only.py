"""User-defined laws with parameter-only coordinates, without a device (extmcmc_user_law_check_theta_only,
DeviceLaw(..., theta_only=...)): every kernel of the program variant compiles without spills in every mode
and chunk width, the argument checks of the C entry points and of the Python constructor, and the
declaration as the law reports it."""
import ctypes as C
import re

import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws_theta as ut

P = ut.G + 2
# 0-based masks of the sample laws' parameter-only coordinates: mu and tau of hier, log lambda of ridge
MASK = {"hier": (1 << (P - 2)) | (1 << (P - 1)), "ridge": 1 << (P - 1)}
COORDS = {"hier": (P - 1, P), "ridge": (P,)}


def _check(src, Pn, D, with_grad, mask, chunk=0, flags=_abi.USER_THETA_TERM):
    buf = C.create_string_buffer(1 << 20)
    used = C.c_int32(-1)
    rc = _abi.load().extmcmc_user_law_check_theta_only(src.encode(), Pn, D, with_grad, chunk, flags, mask,
                                                        C.byref(used), buf, len(buf))
    return rc, used.value, buf.value.decode()


def _kernels(log):
    """entry function -> (spill stores, spill loads, registers)"""
    return {m.group(1): (int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in re.finditer(
        r"Function properties for (extmcmc_user_\w+)\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads\n"
        r".*?Used (\d+) registers", log)}


MODES = [(_abi.USER_GRAD_NONE, 0), (_abi.USER_GRAD_HAND, 0), (_abi.USER_GRAD_FORWARD, 0),
         (_abi.USER_GRAD_FORWARD, 3), (_abi.USER_GRAD_FORWARD, 5)]


@pytest.mark.parametrize("with_grad,chunk", MODES)
@pytest.mark.parametrize("name", list(ut.LAWS))
def test_every_kernel_of_the_variant_compiles_without_spills(name, with_grad, chunk):
    hand, fwd, Df, _, _ = ut.LAWS[name]
    src = fwd if with_grad == _abi.USER_GRAD_FORWARD else hand
    rc, used, log = _check(src, P, Df(P), with_grad, MASK[name], chunk)
    assert rc == _abi.OK, log
    assert used == ((chunk or P) if with_grad == _abi.USER_GRAD_FORWARD else 0)
    ks = _kernels(log)
    # the sweeps of the undeclared program, and the two parameter-only kernels
    theta = {"extmcmc_user_theta_v"} | ({"extmcmc_user_theta_g"} if with_grad else set())
    assert theta <= set(ks), sorted(ks)
    buf = C.create_string_buffer(1 << 20)
    rc0 = _abi.load().extmcmc_user_law_check_ex(src.encode(), P, Df(P), with_grad, chunk or (
        P if with_grad == _abi.USER_GRAD_FORWARD else 0), _abi.USER_THETA_TERM, None, buf, len(buf))
    assert rc0 == _abi.OK
    assert set(ks) == set(_kernels(buf.value.decode())) | theta
    assert all(v[:2] == (0, 0) for v in ks.values()), {k: v for k, v in ks.items() if v[:2] != (0, 0)}


def test_argument_checks_in_c():
    src = ut.HIER_HAND
    # refused before compiling: no flag, an empty declaration, a coordinate at or above n_params
    for mask, flags, what in [(MASK["hier"], 0, "EXTMCMC_USER_THETA_TERM"), (0, _abi.USER_THETA_TERM, "no coordinate"),
                              (1 << P, _abi.USER_THETA_TERM, "n_params"),
                              (MASK["hier"] | (1 << 63), _abi.USER_THETA_TERM, "n_params")]:
        rc, used, log = _check(src, P, 2, _abi.USER_GRAD_HAND, mask, flags=flags)
        assert rc == _abi.EINVAL and used == -1 and what in log, (mask, flags, log)
    # the other arguments as in the _ex entry points
    rc, used, log = _check(src, P, 2, _abi.USER_GRAD_HAND, MASK["hier"], chunk=2)
    assert rc == _abi.EINVAL and used == -1 and "chunk must be 0 unless" in log, log
    rc, used, log = _check(src, P, 2, _abi.USER_GRAD_HAND, MASK["hier"], flags=_abi.USER_THETA_TERM | 2)
    assert rc == _abi.EINVAL and used == -1 and "flags" in log, log
    assert _check(src, 65, 2, _abi.USER_GRAD_HAND, 1)[0] == _abi.EUNSUPPORTED
    # bit 63 is coordinate 64 of a 64-parameter law
    assert _check(ut.RIDGE_POISSON, 64, 63, _abi.USER_GRAD_NONE, 1 << 63)[0] == _abi.OK
    lib = _abi.load()
    assert lib.extmcmc_set_user_law_theta_only(None, src.encode(), 1, 0, _abi.USER_THETA_TERM, MASK["hier"]) == _abi.EINVAL


def test_the_declaration_is_part_of_the_program():
    # a declared law compiles another program than the undeclared one (its own cache entry and log)
    rc, _, log = _check(ut.HIER_HAND, P, 2, _abi.USER_GRAD_HAND, MASK["hier"])
    buf = C.create_string_buffer(1 << 20)
    rc0 = _abi.load().extmcmc_user_law_check_ex(ut.HIER_HAND.encode(), P, 2, _abi.USER_GRAD_HAND, 0,
                                                 _abi.USER_THETA_TERM, None, buf, len(buf))
    assert rc == rc0 == _abi.OK
    assert "extmcmc_user_theta_g" in log and "extmcmc_user_theta" not in buf.value.decode()


def test_device_law_reports_the_declaration():
    law = em.DeviceLaw(ut.HIER_HAND, P, 2, gradient=True, theta_term=True, theta_only=[P, P - 1])
    assert law.theta_only == (P - 1, P) and law.theta_term is True
    assert em.DeviceLaw(ut.HIER_HAND, P, 2, gradient=True, theta_term=True).theta_only is None
    law = em.DeviceLaw(ut.HIER_FORWARD, P, 2, gradient="forward", chunk=3, theta_term=True, theta_only=(P - 1, P))
    assert law.chunk == 3 and law.theta_only == (P - 1, P)
    law = em.DeviceLaw(ut.RIDGE_POISSON, P, P - 1, gradient=True, theta_term=True, theta_only=iter([P]))
    assert law.theta_only == (P,)


@pytest.mark.parametrize("bad,match", [
    ([P, P], "twice"), ([0], "outside"), ([P + 1], "outside"), ([-1], "outside"), ([1.0], "integers"),
    ([True], "integers"), (["1"], "integers"), ([], "no coordinate"), (3, "iterable"), ("12", "iterable")])
def test_device_law_refuses_bad_declarations(bad, match):
    with pytest.raises(ValueError, match=match):
        em.DeviceLaw(ut.HIER_HAND, P, 2, gradient=True, theta_term=True, theta_only=bad)


def test_device_law_needs_the_theta_term():
    with pytest.raises(ValueError, match="theta_term=True"):
        em.DeviceLaw(ut.HIER_HAND, P, 2, gradient=True, theta_only=[P])
