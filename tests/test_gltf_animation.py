"""glTF node animation in the Python loader (gltf.load_gltf(..., time=, animation=)): time=None is the static loader bit
for bit, a key's time is the static file with that key's TRS written into the nodes, and between keys LINEAR, slerp and
STEP follow a float64 statement.  The animated files are written with scenes/gen_gltf.py's builder."""
import json
import os

import numpy as np
import pytest

import gen_gltf
from scene_digest import flattening_digest

from rt_b200 import gltf

SCENES = ["tiny", "texall", "texmaps", "small", "small_lights", "small_manylights"]
F = np.float32

# tiny: node 0 holds the mesh, node 1 the camera (translation [0, 1.6, 2.5], a small rotation about x)
Q_A = np.array([-0.0499792, 0.0, 0.0, 0.9987503], F)
Q_B = (np.array([0.1, 0.7, -0.05, 0.7], np.float64) / np.linalg.norm([0.1, 0.7, -0.05, 0.7])).astype(F)
Q_C = np.array([-0.0, 0.2, -0.0, -0.9797959], F)  # its shortest arc from Q_B flips the sign
MESH_T = ([0.0, 0.5, 1.25, 2.0], [[0, 0, 0], [0.25, -0.0, 0.5], [1.0, 0.125, -0.75], [-0.5, 0.0, 0.0]])
MESH_S = ([0.0, 1.0, 2.0], [[1, 1, 1], [1.5, 0.5, 2.0], [0.75, 1.0, 1.0]])
MESH_R = ([0.0, 1.0, 2.0], [[0, 0, 0, 1], Q_B, Q_C])
CAM_T = ([0.25, 1.5], [[0.0, 1.6, 2.5], [0.5, 1.9, 2.0]])
CAM_R = ([0.25, 1.5], [Q_A, Q_B])


def _animated(name, out_dir, channels):
    g = gen_gltf.SCENES[name]()
    g.animation(channels)
    return g.write(out_dir)


def _tiny_channels():
    return [(0, "translation", *MESH_T, "LINEAR"), (0, "scale", *MESH_S, "STEP"), (0, "rotation", *MESH_R, "LINEAR"),
            (1, "translation", *CAM_T, "LINEAR"), (1, "rotation", *CAM_R, "LINEAR")]


def _same(a, b):
    assert flattening_digest(a) == flattening_digest(b)
    for k in ("tri_pos", "tri_normals", "tri_uv", "tri_tangents"):
        assert getattr(a, k).tobytes() == getattr(b, k).tobytes(), k
    assert a.cameras == b.cameras and a.projections == b.projections


@pytest.mark.parametrize("name", SCENES)
def test_time_none_is_the_static_loader(name, tmp_path):
    static = gen_gltf.generate(name, str(tmp_path / "static"))
    animated = _animated(name, str(tmp_path / "anim"), [(0, "translation", [0.0, 1.0], [[0, 0, 0], [1, 2, 3]], "LINEAR")])
    _same(gltf.load_gltf(static, 1.25), gltf.load_gltf(animated, 1.25))
    _same(gltf.load_gltf(static, 1.25), gltf.load_gltf(gltf.GltfFile(animated), 1.25))


def _static_copy(path, out, time):
    """The animated file with its animation removed and, for every channel, the value of the key at `time` written into
    the target node's TRS (JSON floats of the float32 key values: exact)."""
    with open(path) as f:
        doc = json.load(f)
    src = gltf.GltfFile(path)
    for ch in doc["animations"][0]["channels"]:
        smp = doc["animations"][0]["samplers"][ch["sampler"]]
        times = gltf._float_accessor(src.doc, src.buffers, smp["input"]).reshape(-1)
        values = gltf._float_accessor(src.doc, src.buffers, smp["output"])
        k = int(np.flatnonzero(times.astype(np.float64) == time)[0]) if (times.astype(np.float64) == time).any() else \
            (0 if time < times[0] else len(times) - 1)
        doc["nodes"][ch["target"]["node"]][ch["target"]["path"]] = [float(v) for v in values[k]]
    del doc["animations"]
    with open(out, "w") as f:
        json.dump(doc, f)
    return out


def test_key_times_are_the_static_file_with_that_key(tmp_path):
    path = _animated("tiny", str(tmp_path), _tiny_channels())
    keys = sorted(set(MESH_T[0]) | set(MESH_S[0]) | set(MESH_R[0]) | set(CAM_T[0]) | set(CAM_R[0]))
    # every channel's key at every time that is a key of ALL channels, plus the clamped ends
    common = [t for t in keys if all(t in c[0] or t < c[0][0] or t > c[0][-1] for c in (MESH_T, MESH_S, MESH_R, CAM_T, CAM_R))]
    assert common  # 0.0 (camera clamped to its first key) and 2.0 (translation and camera clamped to their last)
    for t in common + [-1.0, 5.0]:
        anim = gltf.load_gltf(path, 1.0, time=t)
        static = gltf.load_gltf(_static_copy(path, str(tmp_path / f"static_{t}.gltf"), t), 1.0)
        _same(anim, static)


def test_negative_zero_survives_a_key(tmp_path):
    path = _animated("tiny", str(tmp_path), [(0, "translation", [0.0, 1.0], [[-0.0, 0.25, -0.0], [1, 1, 1]], "LINEAR")])
    sc = gltf.load_gltf(path, 1.0, time=0.0)
    ref = gltf.load_gltf(_static_copy(path, str(tmp_path / "s.gltf"), 0.0), 1.0)
    _same(sc, ref)


def _f64_linear(times, values, t):
    times = np.asarray(times, F).astype(np.float64)
    values = np.asarray(values, F).astype(np.float64)
    t = min(max(t, times[0]), times[-1])
    k = min(np.searchsorted(times, t, side="right") - 1, len(times) - 2)
    u = (t - times[k]) / (times[k + 1] - times[k])
    return values[k] * (1 - u) + values[k + 1] * u


def _f64_slerp(times, values, t):
    times = np.asarray(times, F).astype(np.float64)
    values = np.asarray(values, F).astype(np.float64)
    t = min(max(t, times[0]), times[-1])
    k = min(np.searchsorted(times, t, side="right") - 1, len(times) - 2)
    u = (t - times[k]) / (times[k + 1] - times[k])
    a, b = values[k], values[k + 1]
    if a @ b < 0:
        b = -b
    th = np.arccos(np.clip(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)), -1, 1))
    q = a * u if th == 0 else (np.sin((1 - u) * th) * a + np.sin(u * th) * b) / np.sin(th)
    return q / np.linalg.norm(q)


@pytest.mark.parametrize("t", [0.1, 0.5 + 1e-3, 0.77, 1.3, 1.999])
def test_between_keys_against_float64(t):
    for times, values in (MESH_T, CAM_T):
        got = gltf.sample_channel(np.asarray(times, F), np.asarray(values, F), "LINEAR", "translation", t)
        ref = _f64_linear(times, values, t)
        assert np.allclose(got, ref, rtol=1e-6, atol=1e-6 * np.abs(ref).max())
    for times, values in (MESH_R, CAM_R):
        got = gltf.sample_channel(np.asarray(times, F), np.asarray(values, F), "LINEAR", "rotation", t)
        ref = _f64_slerp(times, values, t)
        assert np.allclose(got, ref, rtol=1e-6, atol=1e-6) and abs(np.linalg.norm(got.astype(np.float64)) - 1) < 1e-6
    times, values = MESH_S
    got = gltf.sample_channel(np.asarray(times, F), np.asarray(values, F), "STEP", "scale", t)
    k = min(np.searchsorted(np.asarray(times, F).astype(np.float64), t, side="right") - 1, len(times) - 1)
    assert got.tobytes() == np.asarray(values[k], F).tobytes()


def test_slerp_takes_the_shortest_arc():
    """Q_B to Q_C: their dot is negative, so the path goes to -Q_C; half way the result is the normalised sum."""
    times = np.array([0.0, 1.0], F)
    values = np.stack([Q_B, Q_C]).astype(F)
    assert float(Q_B.astype(np.float64) @ Q_C.astype(np.float64)) < 0
    mid = gltf.sample_channel(times, values, "LINEAR", "rotation", 0.5).astype(np.float64)
    ref = Q_B.astype(np.float64) - Q_C.astype(np.float64)
    assert np.allclose(mid, ref / np.linalg.norm(ref), atol=1e-6)


def test_clamping_at_both_ends():
    times, values = np.asarray(MESH_T[0], F), np.asarray(MESH_T[1], F)
    assert gltf.sample_channel(times, values, "LINEAR", "translation", -3.0).tobytes() == values[0].tobytes()
    assert gltf.sample_channel(times, values, "LINEAR", "translation", 99.0).tobytes() == values[-1].tobytes()
    assert gltf.sample_channel(times, values, "STEP", "translation", 99.0).tobytes() == values[-1].tobytes()


def test_animated_camera_moves_the_scene_camera(tmp_path):
    path = _animated("tiny", str(tmp_path), _tiny_channels())
    assert gltf.animation_range(path) == (0.0, 2.0)
    c0 = gltf.load_gltf(path, 1.0, time=0.25).camera()
    c1 = gltf.load_gltf(path, 1.0, time=1.0).camera()
    assert c0 != c1
    # a root camera node's position is its translation exactly
    assert np.allclose(c1.position.astype(np.float64), _f64_linear(*CAM_T, 1.0), rtol=1e-6)
    assert c0.position.tobytes() == np.asarray(CAM_T[1][0], F).tobytes()
    assert gltf.load_gltf(path, 1.0).camera() == gltf.load_gltf(path, 1.0, time=0.25).camera()  # the rest pose is key 0
    # and the ADD_LIGHT_TRIANGLE light, which is placed in the camera's frame, follows it
    a = gltf.load_gltf(path, 1.0, time=0.25, add_light_triangle=True).tri_pos[-1]
    b = gltf.load_gltf(path, 1.0, time=1.0, add_light_triangle=True).tri_pos[-1]
    assert not np.array_equal(a, b)


@pytest.mark.parametrize("what", ["cubicspline", "weights", "skin", "no_animations", "out_of_range"])
def test_unsupported_animation_raises(what, tmp_path):
    if what == "cubicspline":
        path = _animated("tiny", str(tmp_path), [(0, "translation", [0.0, 1.0], [[0, 0, 0]] * 6, "CUBICSPLINE")])
    elif what == "weights":
        path = _animated("tiny", str(tmp_path), [(0, "weights", [0.0, 1.0], [0.0, 1.0], "LINEAR")])
    elif what == "no_animations":
        path = gen_gltf.generate("tiny", str(tmp_path))
    else:
        path = _animated("tiny", str(tmp_path), [(0, "translation", [0.0, 1.0], [[0, 0, 0], [1, 0, 0]], "LINEAR")])
        if what == "skin":
            with open(path) as f:
                doc = json.load(f)
            doc["skins"] = [{"joints": [1]}]
            doc["nodes"][0]["skin"] = 0
            with open(path, "w") as f:
                json.dump(doc, f)
    gltf.load_gltf(path, 1.0)  # without a time the file loads as before
    with pytest.raises(gltf.AnimationError):
        gltf.load_gltf(path, 1.0, time=0.5, animation=1 if what == "out_of_range" else 0)
