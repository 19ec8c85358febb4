"""Adaptive sampling without a GPU: the stopping rule of csrc/adaptive.cuh compiled for the host (the same function
k_adapt_flags evaluates), the new C ABI symbols, and the no-device failure of an adaptive render."""
import ctypes as C
import math
import os
import shutil
import subprocess
import sys

import pytest

from conftest import ROOT

import rt_b200  # noqa: F401
from rt_b200 import _abi, gpu

CSRC = os.path.join(ROOT, "raytracing-course-hw-public_b200", "csrc")

SHIM = r"""
#include "adaptive.cuh"
extern "C" double adapt_rel_error(double s, double q, unsigned n, double abs_floor) { return rt::adapt_rel_error(s, q, n, abs_floor); }
extern "C" double adapt_luma_sum(float r, float g, float b) { return rt::adapt_luma_sum(r, g, b); }
extern "C" int adapt_converged(double err, float rel_error) { return rt::adapt_converged(err, rel_error) ? 1 : 0; }
"""


@pytest.fixture(scope="module")
def rule(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no host C++ compiler")
    d = tmp_path_factory.mktemp("adaptive_rule")
    src, so = d / "shim.cpp", d / "libadaptive_rule.so"
    src.write_text(SHIM)
    subprocess.run([gxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-I" + CSRC, "-o", str(so), str(src)], check=True)
    L = C.CDLL(str(so))
    L.adapt_rel_error.argtypes = [C.c_double, C.c_double, C.c_uint, C.c_double]
    L.adapt_rel_error.restype = C.c_double
    L.adapt_luma_sum.argtypes = [C.c_float, C.c_float, C.c_float]
    L.adapt_luma_sum.restype = C.c_double
    L.adapt_converged.argtypes = [C.c_double, C.c_float]
    return L


def moments(values):
    return sum(values), sum(v * v for v in values), len(values)


@pytest.mark.parametrize("value", [0.0, 0.25, 2.0, 1.5])
@pytest.mark.parametrize("n", [2, 7, 64])
def test_constant_samples_have_no_error(rule, value, n):
    s, q, n = moments([value] * n)
    assert rule.adapt_rel_error(s, q, n, 1e-3) == 0.0


@pytest.mark.parametrize("u,v,a,b,floor", [(0.0, 1.0, 3, 5, 1e-3), (0.2, 3.5, 10, 2, 1e-2), (1.0, 1.25, 1, 1, 1e-3)])
def test_two_valued_samples_match_the_closed_form(rule, u, v, a, b, floor):
    """a samples of u and b of v: mean (a u + b v) / n, unbiased variance a b (u - v)^2 / (n (n - 1))."""
    s, q, n = moments([u] * a + [v] * b)
    m = (a * u + b * v) / n
    var = a * b * (u - v) ** 2 / (n * (n - 1))
    want = math.sqrt(var / n) / (m + floor)
    assert rule.adapt_rel_error(s, q, n, floor) == pytest.approx(want, rel=1e-12)


def test_rule_edges(rule):
    assert math.isinf(rule.adapt_rel_error(1.0, 1.0, 1, 1e-3))  # one sample: no variance estimate, never converged
    assert rule.adapt_luma_sum(3.0, 6.0, 0.0) == 3.0
    assert rule.adapt_converged(0.125, 0.25) == 1 and rule.adapt_converged(0.25, 0.25) == 1  # err <= target
    assert rule.adapt_converged(0.375, 0.25) == 0
    assert rule.adapt_converged(0.0, 0.0) == 0  # target 0: never stops early, even without noise
    assert rule.adapt_converged(float("nan"), 0.5) == 0  # an infinite sample keeps the pixel going


def test_adaptive_symbols_are_exported():
    assert "rt_gpu_render_adaptive" in gpu.SYMBOLS and "rt_gpu_readback_adaptive" in gpu.SYMBOLS
    L = C.CDLL(gpu.LIB_PATH)
    for name in ("rt_gpu_render_adaptive", "rt_gpu_readback_adaptive"):
        getattr(L, name)
    assert C.sizeof(_abi.rt_adaptive_params) == 16
    assert C.sizeof(_abi.rt_render_params) == 48  # unchanged


def test_adaptive_render_fails_without_a_device():
    """In a child process that sees no device (so that this runs on a GPU machine as well)."""
    code = ("import sys; sys.path.insert(0, sys.argv[1]); import rt_b200; from rt_b200 import gpu\n"
            "try:\n    gpu.RtGpu(1, 0).render_adaptive(8, 8, 16, 4, 4, 0.05)\n"
            "except gpu.RtGpuError as e:\n    print(e)\n    sys.exit(0)\nsys.exit(1)\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and "RT_ERR_NO_DEVICE" in r.stdout, r.stdout + r.stderr
