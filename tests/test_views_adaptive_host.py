"""Adaptive multi-view rendering without a GPU: the new C ABI symbol, its null-argument check, the no-device failure
through the Python method, and the unchanged structs."""
import ctypes as C
import os
import subprocess
import sys

import pytest

from conftest import ROOT

import rt_b200
from rt_b200 import _abi, gpu

NAME = "rt_gpu_render_views_adaptive"


def test_symbol_is_exported_and_declared():
    assert NAME in gpu.SYMBOLS
    getattr(C.CDLL(gpu.LIB_PATH), NAME)
    with open(os.path.join(ROOT, "include", "rt_gpu.h")) as f:
        assert f"int {NAME}(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views," in f.read()


def test_null_arguments_are_refused_before_any_device_work():
    """Every argument is checked before the handle is used: this runs on a machine without a GPU."""
    L = gpu.lib()
    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    cams = (_abi.rt_camera * 1)(rt_b200.Camera([0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0).to_c())
    p = _abi.rt_render_params(8, 8, 16, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, 0, 0, 0)
    v = _abi.rt_views(1, 0, cams)
    a = _abi.rt_adaptive_params(4, 4, 0.05, 1e-3)
    assert L.rt_gpu_render_views_adaptive(None, C.byref(p), C.byref(v), C.byref(a)) == bad
    assert L.rt_gpu_render_views_adaptive(None, None, None, None) == bad
    assert NAME in L.rt_gpu_last_error().decode()


def test_struct_sizes_are_unchanged():
    assert C.sizeof(_abi.rt_views) == 16 and C.sizeof(_abi.rt_adaptive_params) == 16
    assert C.sizeof(_abi.rt_camera) == 52 and C.sizeof(_abi.rt_render_params) == 48
    assert C.sizeof(_abi.rt_stats) == 120
    assert _abi.RT_GPU_ABI_VERSION == 1


@pytest.mark.parametrize("via", ["python", "c"])
def test_fails_without_a_device(via):
    """In a child process that sees no device (so that this runs on a GPU machine as well): the Python method raises
    RT_ERR_NO_DEVICE, and so does the C sequence up to the call."""
    if via == "python":
        code = ("import sys; sys.path.insert(0, sys.argv[1]); import rt_b200; from rt_b200 import gpu\n"
                "cam = rt_b200.Camera([0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0)\n"
                "try:\n    gpu.RtGpu(1, 0).render_views_adaptive([cam, cam], 8, 8, 16, 4, 4, 0.05)\n"
                "except gpu.RtGpuError as e:\n    print(e)\n    sys.exit(0)\nsys.exit(1)\n")
    else:
        code = ("import sys, ctypes as C; sys.path.insert(0, sys.argv[1]); import rt_b200; from rt_b200 import _abi, gpu\n"
                "L = gpu.lib(); h = C.c_void_p()\n"
                "rc = L.rt_gpu_create(C.byref(h), 1, 0)\n"
                "if rc == 0:\n    sys.exit(1)\n"
                "print(_abi.STATUS[rc], L.rt_gpu_last_error().decode())\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and "RT_ERR_NO_DEVICE" in r.stdout, r.stdout + r.stderr
