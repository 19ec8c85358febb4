"""Animated geometry without a GPU: the rt_gpu_update_geometry symbol, its struct against the header, the null-argument
check, and the Python CLI's RT_FRAMES refusals (all decided before any device work)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT

import gen_gltf
from rt_b200 import _abi, cli, gpu

NAME = "rt_gpu_update_geometry"


def test_symbol_is_exported_and_declared():
    assert NAME in gpu.SYMBOLS
    getattr(C.CDLL(gpu.LIB_PATH), NAME)
    with open(os.path.join(ROOT, "include", "rt_gpu.h")) as f:
        assert f"int {NAME}(rt_gpu_ctx *ctx, const rt_geometry_update *u);" in f.read()


def test_struct_matches_the_header(tmp_path):
    """sizeof and offsetof of every field, as a C compiler lays out include/rt_gpu.h, against the ctypes mirror."""
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in _abi.rt_geometry_update._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rt_gpu.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(rt_geometry_update));\n' +
                   "".join(f'    printf("%zu\\n", offsetof(rt_geometry_update, {f}));\n' for f in fields) + "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(_abi.rt_geometry_update)] + [getattr(_abi.rt_geometry_update, f).offset for f in fields]
    assert got[0] == 64


def test_null_arguments_are_refused_before_any_device_work():
    L = gpu.lib()
    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    u = _abi.rt_geometry_update()
    assert L.rt_gpu_update_geometry(None, C.byref(u)) == bad
    assert L.rt_gpu_update_geometry(None, None) == bad
    assert NAME in L.rt_gpu_last_error().decode()


def _static_tiny(tmp_path):
    return gen_gltf.generate("tiny", str(tmp_path))


def _animated_tiny(tmp_path):
    g = gen_gltf.tiny()
    g.animation([(0, "translation", [0.0, 1.0], [[0, 0, 0], [0.5, 0, 0]], "LINEAR")])
    return g.write(str(tmp_path))


@pytest.mark.parametrize("case", ["cameras_all", "text_scene", "no_animation", "bad_count", "bad_fps", "no_colon", "bad_animation",
                                  "animation_out_of_range"])
def test_cli_refuses_bad_frames(case, tmp_path, monkeypatch, capsys):
    scene = _animated_tiny(tmp_path)
    env = {"RT_FRAMES": "3:24"}
    if case == "cameras_all":
        env["RT_CAMERAS"] = "all"
    elif case == "text_scene":
        scene = str(tmp_path / "scene.txt")
        with open(scene, "w") as f:
            f.write("DIMENSIONS 8 8\nBG_COLOR 0 0 0\nCAMERA_POSITION 0 0 5\nCAMERA_RIGHT 1 0 0\nCAMERA_UP 0 1 0\n"
                    "CAMERA_FORWARD 0 0 -1\nCAMERA_FOV_X 1.0\n")
    elif case == "no_animation":
        scene = _static_tiny(tmp_path / "static")
    else:
        env["RT_FRAMES"] = {"bad_count": "0:24", "bad_fps": "3:0", "no_colon": "3", "bad_animation": "3:24",
                            "animation_out_of_range": "3:24"}[case]
        if case == "bad_animation":
            env["RT_ANIMATION"] = "first"
        if case == "animation_out_of_range":
            env["RT_ANIMATION"] = "1"
    for k in ("RT_CAMERAS", "RT_ANIMATION", "RT_ADAPTIVE", "RT_PROJECTION"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    out = tmp_path / "out.ppm"
    assert cli.main(["rt", scene, "8", "8", "4", str(out)]) == 1
    assert "RT_FRAMES" in capsys.readouterr().err
    assert not any(p.suffix == ".ppm" for p in tmp_path.iterdir())


def test_parse_frames():
    assert cli.parse_frames("3:24") == (3, 24.0)
    assert cli.parse_frames("1:0.5") == (1, 0.5)
    for bad in ("", "3", "3:", ":24", "-1:24", "3:-1", "3:inf", "3:nan", "x:24", "3:24:1"):
        with pytest.raises(ValueError):
            cli.parse_frames(bad)


def test_geometry_update_aliases_the_scene(golden_scene):
    sc = golden_scene("tiny")
    u = sc.geometry_update()
    assert u.n_tris == sc.n_tris and u.tri_pos == sc.tri_pos.ctypes.data and u.tri_normals == sc.tri_normals.ctypes.data
    assert u.light_bvh.n_objects == len(sc.light_bvh.objects)
    assert (u.tri_tangents or 0) == (sc.tri_tangents.ctypes.data if sc.tri_tangents is not None and sc.tri_tangents.size else 0)
    assert np.asarray(sc.tri_pos).dtype == np.float32
