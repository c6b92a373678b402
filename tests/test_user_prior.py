"""User-defined priors (DevicePrior, EXTMCMC_PRIOR_USER) without a GPU: the NVRTC program of every sample
prior compiles for sm_100a without spills, bad sources and limits are refused, a DevicePrior cannot be a
ProductPrior factor, and the lean step kernels (cfg 2 / 3 / 4) are the instructions they were."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest

import extensiblemcmc_jl_b200 as em
from extensiblemcmc_jl_b200 import _abi
from tests import user_priors as up

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check(src, p_u, with_grad):
    buf = C.create_string_buffer(1 << 16)
    rc = _abi.load().extmcmc_user_prior_check(src.encode(), p_u, with_grad, buf, len(buf))
    return rc, buf.value.decode()


@pytest.mark.parametrize("name,src,with_grad,p_u", [
    ("uniform", up.UNIFORM, _abi.USER_GRAD_NONE, 1), ("uniform", up.UNIFORM, _abi.USER_GRAD_NONE, 8),
    ("uniform", up.UNIFORM, _abi.USER_GRAD_NONE, 32), ("laplace", up.LAPLACE, _abi.USER_GRAD_HAND, 1),
    ("laplace", up.LAPLACE, _abi.USER_GRAD_HAND, 32), ("normal", up.NORMAL, _abi.USER_GRAD_HAND, 1),
    ("normal_forward", up.NORMAL_FORWARD, _abi.USER_GRAD_FORWARD, 16),
    ("student_t_forward", up.STUDENT_T_FORWARD, _abi.USER_GRAD_FORWARD, 16)])
def test_sample_priors_compile_without_spills(name, src, with_grad, p_u):
    rc, log = _check(src, p_u, with_grad)
    assert rc == _abi.OK, log
    spills = [int(s) for s in re.findall(r"(\d+) bytes spill stores", log)]
    assert spills and all(s == 0 for s in spills), log


def test_every_sample_prior_compiles():
    for src, g, p_u in [(up.NORMAL, 1, 2), (up.NORMAL_FORWARD, 2, 2), (up.GAMMA, 0, 2), (up.UNIFORM, 0, 2),
                        (up.BETA, 0, 2), (up.CAUCHY, 0, 2), (up.IMPROPER_POS, 0, 2),
                        (up.PRODUCT_NORMAL_GAMMA, 0, 2), (up.LAPLACE, 1, 64)]:
        rc, log = _check(src, p_u, g)
        assert rc == _abi.OK, log


def test_bad_source_raises_with_the_log():
    with pytest.raises(ValueError, match="undefined_thing"):
        em.DevicePrior(up.BAD)
    with pytest.raises(ValueError, match="logprior_grad"):
        em.DevicePrior(up.UNIFORM, gradient=True)   # no logprior_grad in the source
    with pytest.raises(ValueError):
        em.DevicePrior(up.UNIFORM, gradient="backward")


def test_limits_are_unsupported():
    assert _check(up.UNIFORM, 65, _abi.USER_GRAD_NONE)[0] == _abi.EUNSUPPORTED
    assert _check(up.LAPLACE, 65, _abi.USER_GRAD_HAND)[0] == _abi.EUNSUPPORTED
    assert _check(up.NORMAL_FORWARD, 17, _abi.USER_GRAD_FORWARD)[0] == _abi.EUNSUPPORTED
    assert _check(up.UNIFORM, 0, _abi.USER_GRAD_NONE)[0] == _abi.EUNSUPPORTED


def test_device_prior_to_abi_and_not_a_product_factor():
    p = em.DevicePrior(up.LAPLACE, gradient=True, params=(0.0, 0.5))
    kind, pp = p.to_abi()
    assert kind == _abi.PRIOR_USER and list(pp) == [0.0, 0.5]
    with pytest.raises(NotImplementedError):
        em.ProductPrior([p, em.Normal()], [1, 1]).to_abi()
    # the closed families stay closed
    with pytest.raises(NotImplementedError):
        em.StandardPrior(object()).to_abi()


def _golden():
    path = os.path.join(ROOT, "tests", "golden", "lean_sass_step_kernels.txt")
    lines = [ln.split() for ln in open(path) if ln.strip() and not ln.startswith("#")]
    version = re.search(r"V[\d.]+", open(path).read()).group(0)
    return version, {name: digest for digest, name in lines}


def test_lean_step_kernels_keep_their_sass():
    obj = os.path.join(ROOT, "extensiblemcmc.jl_b200", "csrc", "build", "step_kernels.o")
    if not os.path.exists(obj) or not shutil.which("cuobjdump") or not shutil.which("nvcc"):
        pytest.skip("needs the built step kernels and the CUDA toolkit")
    version, want = _golden()
    have_version = re.search(r"V[\d.]+", subprocess.run(["nvcc", "--version"], capture_output=True, text=True).stdout)
    if not have_version or have_version.group(0) != version:
        pytest.skip(f"the recorded SASS is of nvcc {version}")
    import importlib.util
    spec = importlib.util.spec_from_file_location("lean_sass", os.path.join(ROOT, "tools", "lean_sass.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.lean_sass(obj) == want
