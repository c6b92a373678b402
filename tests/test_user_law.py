"""User-defined device laws without a device: extmcmc_user_law_check compiles the user's source with
the sweep template for sm_100a (NVRTC), and rejects what does not compile with the compiler's log."""
import ctypes as C
import re

import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_laws as ul


def _check(src, P, D, grad):
    buf = C.create_string_buffer(1 << 16)
    rc = _abi.load().extmcmc_user_law_check(src.encode(), P, D, 1 if grad else 0, buf, len(buf))
    return rc, buf.value.decode()


# the three sample laws at the shapes the GPU tests run, with the gradient
@pytest.mark.parametrize("name,P,D", [("gsn1d", 2, 1), ("logistic", 8, 9), ("logistic", 2, 3),
                                      ("poisson_reg", 8, 8), ("poisson_reg", 3, 3), ("poisson_reg", 1, 1)])
def test_sample_laws_compile_without_spills(name, P, D):
    rc, log = _check(ul.LAWS[name][0], P, D, True)
    assert rc == _abi.OK, log
    kernels = re.findall(r"Compiling entry function '(extmcmc_user_\w+)'", log)
    # every instantiation the planner can pick: chains R = 1 (, 2, 4) and lanes, without and with GRAD
    rmax = 4 if (2 * P + 1) * 4 <= 40 else 2 if (2 * P + 1) * 2 <= 40 else 1
    expect = {f"extmcmc_user_chains_r{r}_g{g}" for r in (1, 2, 4) if r <= rmax for g in (0, 1)}
    expect |= {"extmcmc_user_lanes_g0", "extmcmc_user_lanes_g1"}
    assert set(kernels) == expect, kernels
    spills = [int(v) for v in re.findall(r"(\d+) bytes spill (?:stores|loads)", log)]
    assert spills and max(spills) == 0, log
    assert "sm_100a" in log


# the 64 x 64 shape limit (kUserMaxParams = kUserMaxObsDim = 64), with the gradient.  Known cost: the
# gradient kernels spill (theta, the Law and the gradient do not fit the 255 registers of a thread;
# ~1 KB of spill stores, ~3 KB of loads); the plain kernels do not.  The values are checked on the
# device in test_gpu_user_law_kernels.py::test_shape_limit_64.
@pytest.mark.parametrize("name,P,D", [("poisson_reg", 64, 64), ("logistic", 63, 64)])
def test_sample_laws_compile_at_the_shape_limit(name, P, D):
    rc, log = _check(ul.LAWS[name][0], P, D, True)
    assert rc == _abi.OK, log
    blocks = re.findall(r"Compiling entry function '(extmcmc_user_\w+)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads",
                        log, re.S)
    spills = {k: (int(st), int(ld)) for k, st, ld in blocks}
    # P = 64: the accumulators of even one extra chain per thread do not fit, R = 1 only
    assert set(spills) == {"extmcmc_user_chains_r1_g0", "extmcmc_user_chains_r1_g1",
                           "extmcmc_user_lanes_g0", "extmcmc_user_lanes_g1"}, log
    for k, s in spills.items():
        if k.endswith("_g0"):
            assert s == (0, 0), (k, s)
    assert "sm_100a" in log


def test_law_without_gradient_compiles_only_the_plain_kernels():
    rc, log = _check(ul.POISSON_RATE, 1, 1, False)
    assert rc == _abi.OK, log
    assert "_g1" not in log and "extmcmc_user_lanes_g0" in log


def test_cached_compile_returns_the_same_log():
    a = _check(ul.GSN1D, 2, 1, False)
    b = _check(ul.GSN1D, 2, 1, False)
    assert a == b and a[0] == _abi.OK


@pytest.mark.parametrize("src,grad,needle", [
    (ul.GSN1D.replace("L.h = 0.5 / var;", "L.h = 0.5 / var"), False, "law("),   # syntax error: its line
    (ul.GSN1D.split("__device__ double logpdf(")[0], False, "logpdf"),          # no logpdf
    (ul.POISSON_RATE, True, "logpdf_grad"),                                     # gradient promised, missing
])
def test_bad_sources_are_einval_with_the_compiler_log(src, grad, needle):
    rc, log = _check(src, 2 if "th[1]" in src else 1, 1, grad)
    assert rc == _abi.EINVAL
    assert "error" in log and needle in log, log


def test_syntax_error_names_the_users_line():
    bad = "struct Law { double a; };\n__device__ bool set_parameters(Law &L, const double *th) { L.a = th[0] return true; }\n"
    rc, log = _check(bad, 1, 1, False)
    assert rc == _abi.EINVAL
    assert re.search(r"law\(2\): error", log), log


def test_shape_limits():
    assert _check(ul.POISSON_RATE, 0, 1, False)[0] == _abi.EUNSUPPORTED
    assert _check(ul.POISSON_RATE, 1, 65, False)[0] == _abi.EUNSUPPORTED


def test_device_law_construction():
    law = em.DeviceLaw(ul.POISSON_REG, 3, 3, gradient=True)
    assert (law.abi_law(), law.n_params, law.obs_dim, law.abi_y()) == (_abi.LAW_USER, 3, 3, None)
    assert "bytes spill" in law.log
    with pytest.raises(ValueError, match="error"):
        em.DeviceLaw("struct Law {};", 1, 1)
    with pytest.raises(ValueError):
        em.DeviceLaw(ul.POISSON_RATE, 1, 1, gradient=True)


def _create(**kw):
    cfg = _abi.Config()
    cfg.abi_version = _abi.ABI_VERSION
    cfg.n_chains, cfg.n_params, cfg.n_updates, cfg.history_window = 8, 2, 1, 4
    cfg.law, cfg.obs_dim, cfg.world_size = _abi.LAW_USER, 1, 1
    for k, v in kw.items():
        setattr(cfg, k, v)
    h = _abi.Handle()
    lib = _abi.load()
    rc = lib.extmcmc_create(C.byref(cfg), C.byref(h))
    if rc == _abi.OK:
        lib.extmcmc_destroy(h)
    return rc, lib.extmcmc_last_error(None).decode()


def test_create_rejects_what_user_laws_do_not_support():
    # checked before any device is touched
    rc, msg = _create(shard_mode=_abi.SHARD_OBS, world_size=2, rank=0)
    assert rc == _abi.EUNSUPPORTED and "SHARD_OBS" in msg
    assert _create(obs_dim=65)[0] == _abi.EUNSUPPORTED
    assert _create(n_params=65)[0] == _abi.EUNSUPPORTED


def test_set_user_law_needs_a_handle():
    assert _abi.load().extmcmc_set_user_law(None, ul.GSN1D.encode(), 0) == _abi.EINVAL
