"""Chunked forward-mode gradients of user-defined laws without a device
(extmcmc_user_law_check_chunked, DeviceLaw(..., gradient="forward", chunk=...)): at K = P the program is
byte for byte the unchunked one, the sample laws compile at large P with one forward kernel per
(mapping, chunk), the width rule and its errors, and the Python constructor."""
import ctypes as C
import re

import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws_chunked as uc
from tests import user_laws_forward as uf


def _check(src, P, D, chunk):
    buf = C.create_string_buffer(1 << 20)
    used = C.c_int32(-1)
    rc = _abi.load().extmcmc_user_law_check_chunked(src.encode(), P, D, chunk, C.byref(used), buf, len(buf))
    return rc, used.value, buf.value.decode()


def _check_forward(src, P, D):
    buf = C.create_string_buffer(1 << 20)
    rc = _abi.load().extmcmc_user_law_check(src.encode(), P, D, _abi.USER_GRAD_FORWARD, buf, len(buf))
    return rc, buf.value.decode()


def auto_chunk(P):
    """The library's width, restated here only to check it: K = P up to 16, else the balanced split
    into chunks of at most 5."""
    if P <= 16:
        return P
    n = -(-P // 5)
    return -(-P // n)


def _kernels(log):
    """entry function -> (spill stores, spill loads, registers)"""
    return {m.group(1): (int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in re.finditer(
        r"Function properties for (extmcmc_user_\w+)\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads\n"
        r".*?Used (\d+) registers", log)}


def _rmax(P, K):
    n = (P + 1) * (K + 1)
    return 4 if 4 * n <= 40 else 2 if 2 * n <= 40 else 1


@pytest.mark.parametrize("P", [1, 3, 8, 16])
def test_width_p_is_the_unchunked_program(P):
    rc0, log0 = _check_forward(uf.POISSON_REG, P, P)
    for chunk in (P, 0):
        rc, used, log = _check(uf.POISSON_REG, P, P, chunk)
        assert (rc, used) == (rc0, P) and log == log0


# the laws whose fields copy theta compile without spills at the library's width; POS_REG (every field
# a live tangent: P (K + 1) doubles per chain) does not fit the register file above P = 16 at any width
SPILL_FREE = ("poisson_reg", "logistic", "gauss_reg", "gauss_reg_scale")
SHAPES = [(name, min(P, uc.max_params(name))) for name in uc.LAWS for P in (17, 24, 33, 48, 64)]


@pytest.mark.parametrize("name,P", SHAPES)
def test_sample_laws_compile_at_the_library_width(name, P):
    src, Df, _ = uc.LAWS[name]
    rc, K, log = _check(src, P, Df(P), 0)
    assert rc == _abi.OK, log
    assert K == auto_chunk(P)
    nc = -(-P // K)
    assert 1 < nc <= 16 and (nc - 1) * K < P
    ks = _kernels(log)
    rs = [r for r in (1, 2, 4) if r <= _rmax(P, K)]
    expect = {f"extmcmc_user_chains_r{r}_g0" for r in rs} | {"extmcmc_user_lanes_g0"}
    expect |= {f"extmcmc_user_chains_r{r}_f{K}c{c}" for r in rs for c in range(nc)}
    expect |= {f"extmcmc_user_lanes_f{K}c{c}" for c in range(nc)}
    assert set(ks) == expect, sorted(set(ks) ^ expect)
    print(name, P, K, nc, "registers", max(v[2] for v in ks.values()), "spill", max(v[0] for v in ks.values()))
    if name in SPILL_FREE:
        assert all(v[:2] == (0, 0) for v in ks.values()), {k: v for k, v in ks.items() if v[:2] != (0, 0)}


def test_explicit_width_and_ragged_last_chunk():
    rc, used, log = _check(uf.POISSON_REG, 20, 20, 7)      # chunks of 7, 7, 6
    assert (rc, used) == (_abi.OK, 7), log
    assert set(k for k in _kernels(log) if "_f" in k) == {
        f"extmcmc_user_{m}_f7c{c}" for m in ("chains_r1", "lanes") for c in range(3)}
    # at P <= 16 a narrower width chunks too, and may plan more chains per thread: (4)(2) doubles -> R = 4
    rc, used, log = _check(uf.POISSON_REG, 3, 3, 1)
    assert (rc, used) == (_abi.OK, 1), log
    assert {"extmcmc_user_chains_r4_f1c2", "extmcmc_user_chains_r4_g0", "extmcmc_user_lanes_f1c0"} <= set(_kernels(log))


@pytest.mark.parametrize("P,chunk", [(20, -1), (20, 17), (8, 9), (1, 2), (64, 3), (33, 2), (17, 1)])
def test_bad_widths_are_einval(P, chunk):
    rc, used, log = _check(uf.POISSON_REG, P, P, chunk)
    assert rc == _abi.EINVAL and used == -1, (rc, log)
    assert "chunk" in log and "chunk" in _abi.load().extmcmc_last_error(None).decode()


def test_widths_at_the_limits():
    # 16 chunks is the most: P = 64 at K = 4, P = 17 at K = 2
    for P, K in ((64, 4), (17, 2), (64, 16), (17, 16)):
        rc, used, log = _check(uf.POISSON_REG, P, P, K)
        assert (rc, used) == (_abi.OK, K), log
    # more than 64 parameters: unsupported, as for every user law
    assert _check(uf.POISSON_REG, 65, 64, 0)[0] == _abi.EUNSUPPORTED
    assert _check(uf.POISSON_REG, 0, 1, 0)[0] == _abi.EUNSUPPORTED
    # a source that does not compile: EINVAL with the log, after the width was resolved
    rc, used, log = _check(uf.BAD_LGAMMA, 1, 1, 0)
    assert rc == _abi.EINVAL and used == 1 and "lgamma" in log
    rc, used, log = _check(uf.BAD_NARROW, 1, 1, 1)
    assert rc == _abi.EINVAL and "const double lam" in log


def test_the_unchunked_entry_point_keeps_its_limit():
    buf = C.create_string_buffer(1 << 12)
    rc = _abi.load().extmcmc_user_law_check(uf.POISSON_REG.encode(), 17, 17, _abi.USER_GRAD_FORWARD, buf, len(buf))
    assert rc == _abi.EUNSUPPORTED and "n_params <= 16" in buf.value.decode()
    assert "extmcmc_set_user_law_chunked" in buf.value.decode()


def test_device_law_chunk_argument():
    law = em.DeviceLaw(uf.POISSON_REG, 24, 24, gradient="forward", chunk="auto")
    assert (law.chunk, law.gradient, law.n_params) == (5, "forward", 24)
    assert "extmcmc_user_lanes_f5c4" in law.log
    assert em.DeviceLaw(uf.POISSON_REG, 24, 24, gradient="forward", chunk=8).chunk == 8
    assert em.DeviceLaw(uf.POISSON_REG, 5, 5, gradient="forward", chunk="auto").chunk == 5
    assert em.DeviceLaw(uf.POISSON_REG, 5, 5, gradient="forward").chunk == 5
    from tests import user_laws as ul
    assert em.DeviceLaw(ul.POISSON_REG, 5, 5, gradient=True).chunk is None
    # chunk=None keeps the unchunked limit
    with pytest.raises(_abi.ExtMCMCError) as ei:
        em.DeviceLaw(uf.POISSON_REG, 17, 17, gradient="forward")
    assert ei.value.code == _abi.EUNSUPPORTED
    # a chunk without forward mode, or not a width
    for grad in (False, True):
        with pytest.raises(ValueError, match="chunk needs gradient='forward'"):
            em.DeviceLaw(ul.POISSON_REG, 5, 5, gradient=grad, chunk=2)
    for bad in (0, -3, True, 2.0, "Auto", "4", [4]):
        with pytest.raises(ValueError, match="chunk must be"):
            em.DeviceLaw(uf.POISSON_REG, 5, 5, gradient="forward", chunk=bad)
    # widths the library refuses
    for P, bad in ((20, 17), (5, 6), (64, 3)):
        with pytest.raises(ValueError, match="chunk"):
            em.DeviceLaw(uf.POISSON_REG, P, P, gradient="forward", chunk=bad)
    with pytest.raises(ValueError, match="does not compile"):
        em.DeviceLaw(uf.BAD_LGAMMA, 1, 1, gradient="forward", chunk="auto")


def test_set_user_law_chunked_needs_a_handle():
    assert _abi.load().extmcmc_set_user_law_chunked(None, uf.GSN1D.encode(), 0) == _abi.EINVAL
