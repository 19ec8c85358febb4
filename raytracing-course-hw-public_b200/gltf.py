"""Host-side glTF loader: a float32-exact mirror of the reference's `parse_gltf_scene`
(src/scene.h:183-501) that produces the flattened `SceneData` directly.

It exists so that hosts without the reference headers (Python, the GPU box) can build the same scene the
reference-hosted flattener (host/flatten_ref.hpp) produces; tests compare the two bit for bit.  The
reference's quirks are kept on purpose because they change the image:
  * accessor byteOffset / bufferView byteStride are ignored for vertex attributes (scene.h:118-133),
    honoured (byteOffset only) for indices (scene.h:142-181);
  * the tangent attribute is looked up as lowercase "tangent" (scene.h:336) and used raw;
  * normals go through `rs_fast_inv_t` (geometry.h:303-311), positions through the full 4x4;
  * node transform = parent * matrix * T*R*S even when both are given (scene.h:228-230);
  * fov_x = 2*atan(tan(yfov/2) * aspect), aspect from the camera or W/H (scene.h:238-254);
  * every material gets ior 1.5; emissive strength extension multiplies the factor (scene.h:263-278).
All arithmetic is done in float32 in the reference's operation order; tan/atan come from libm (tanf/atanf)
because the reference calls exactly those.
"""
import ctypes
import ctypes.util
import json
import os

import numpy as np

from . import host
from ._abi import MATERIAL_DTYPE, TEXTURE_DTYPE, Camera, Projection, SceneData

F = np.float32
_libm = ctypes.CDLL(ctypes.util.find_library("m") or "libm.so.6")
for _fn in ("tanf", "atanf"):
    getattr(_libm, _fn).restype = ctypes.c_float
    getattr(_libm, _fn).argtypes = [ctypes.c_float]


def tanf(x):
    return F(_libm.tanf(float(x)))


def atanf(x):
    return F(_libm.atanf(float(x)))


def _mat_mul(a, b):
    """matrix4 operator*, geometry.h:216-228: res[i][k] += a[i][j]*b[j][k], j ascending, float32."""
    res = np.zeros((4, 4), F)
    for i in range(4):
        for j in range(4):
            for k in range(4):
                res[i, k] = F(res[i, k] + F(a[i, j] * b[j, k]))
    return res


def _translation(t):
    m = np.eye(4, dtype=F)
    m[0, 3], m[1, 3], m[2, 3] = t
    return m


def _scale(s):
    m = np.eye(4, dtype=F)
    m[0, 0], m[1, 1], m[2, 2] = s
    return m


def _rotation(q):
    """matrix4::rotation, geometry.h:179-196; q = (x, y, z, w)."""
    x, y, z, w = (F(v) for v in q)
    two, one = F(2), F(1)
    m = np.eye(4, dtype=F)
    m[0, :3] = [one - two * (y * y + z * z), two * (x * y - z * w), two * (x * z + y * w)]
    m[1, :3] = [two * (x * y + z * w), one - two * (x * x + z * z), two * (y * z - x * w)]
    m[2, :3] = [two * (x * z - y * w), two * (y * z + x * w), one - two * (x * x + y * y)]
    return m


def _parse_mat4(src):
    """parse_mat4, scene.h:101-108: glTF column-major -> row-major."""
    return np.array([[src[0], src[4], src[8], src[12]], [src[1], src[5], src[9], src[13]],
                     [src[2], src[6], src[10], src[14]], [src[3], src[7], src[11], src[15]]], F)


def _normal_matrix(m4):
    """matrix3(transform).rs_fast_inv_t(), geometry.h:287-311."""
    m = m4[:3, :3]
    d2 = F(F(_len2(m[0]) * _len2(m[1])) * _len2(m[2]))
    res = np.zeros((3, 3), F)
    for r in range(3):
        for c in range(3):
            r1, r2, c1, c2 = (r + 1) % 3, (r + 2) % 3, (c + 1) % 3, (c + 2) % 3
            res[r, c] = F(F(F(m[r1, c1] * m[r2, c2]) - F(m[r1, c2] * m[r2, c1])) / d2)
    return res


def _len2(v):
    return F(F(F(v[0] * v[0]) + F(v[1] * v[1])) + F(v[2] * v[2]))


def _apply_points(m, p):
    """matrix4::apply, geometry.h:259-261: dot(row, (x, y, z, 1)) left to right."""
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    out = np.empty_like(p)
    for i in range(3):
        out[:, i] = ((m[i, 0] * x + m[i, 1] * y) + m[i, 2] * z) + m[i, 3] * F(1)
    return out


def _apply_normals(m3, n):
    """norm(normal_transform.apply(n)), scene.h:392-397."""
    x, y, z = n[:, 0], n[:, 1], n[:, 2]
    out = np.empty_like(n)
    for i in range(3):
        out[:, i] = (m3[i, 0] * x + m3[i, 1] * y) + m3[i, 2] * z
    return _normalize(out)


def _normalize(v):
    ln = np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])
    with np.errstate(divide="ignore", invalid="ignore"):
        return v / ln[:, None]


def _load_texture(path):
    """Texture::load_img, geometry.h:584-598 (stb_image forced to 4 x 8 bit)."""
    from PIL import Image

    with Image.open(path) as im:
        rgba = np.asarray(im.convert("RGBA"), np.uint8)
    return np.ascontiguousarray(rgba)


_COMPONENT = {5121: np.uint8, 5123: np.uint16, 5125: np.uint32}


# config.h:39-47: the extra light source, in camera coordinates (right, up, forward)
LIGHT_TRIANGLE_INTENSITY = 10.0
LIGHT_TRIANGLE_RELATIVE_POS = ((10.0, 0.0, -0.1), (0.0, 10.0, -0.1), (0.0, -10.0, -0.1))


class AnimationError(ValueError):
    """An animation the loader cannot sample (see load_gltf's `time`)."""


def _read_buffers(doc, base):
    buffers = []
    for b in doc.get("buffers", []):
        raw = np.zeros(int(b["byteLength"]), np.uint8)
        with open(os.path.join(base, b["uri"]), "rb") as f:
            data = np.frombuffer(f.read(int(b["byteLength"])), np.uint8)
        raw[:data.size] = data
        buffers.append(raw)
    return buffers


_COMPS = {"SCALAR": 1, "VEC2": 2, "VEC3": 3, "VEC4": 4}


def _float_accessor(doc, buffers, idx):
    """A float accessor as the glTF specification lays it out (bufferView and accessor byteOffset, byteStride):
    [count, components] float32.  Animation data only; vertex attributes keep the reference's reading."""
    acc = doc["accessors"][idx]
    if int(acc["componentType"]) != 5126:
        raise AnimationError(f"accessor {idx}: animation data must be float (componentType 5126)")
    view = doc["bufferViews"][int(acc["bufferView"])]
    comps, count = _COMPS[acc["type"]], int(acc["count"])
    stride = int(view.get("byteStride", 4 * comps))
    off = int(view.get("byteOffset", 0)) + int(acc.get("byteOffset", 0))
    buf = buffers[int(view["buffer"])]
    out = np.empty((count, comps), F)
    for k in range(count):
        out[k] = buf[off + k * stride:off + k * stride + 4 * comps].view(F)
    return out


def _animation(doc, animation):
    anims = doc.get("animations") or []
    if not anims:
        raise AnimationError("the file has no animations")
    if not 0 <= animation < len(anims):
        raise AnimationError(f"animation {animation} out of range: the file has {len(anims)}")
    return anims[animation]


class GltfFile:
    """A glTF file read once: its JSON, buffers and texture images (images are decoded on first use and kept), so that
    many frames of an animation can be flattened from one read (load_gltf and animation_range take one for a path)."""

    def __init__(self, path):
        self.path = path
        with open(path) as f:
            self.doc = json.load(f)
        self.base = os.path.dirname(os.path.abspath(path))
        self.buffers = _read_buffers(self.doc, self.base)
        self._images = {}

    def image(self, path):
        if path not in self._images:
            self._images[path] = _load_texture(path)
        return self._images[path]

    def textures(self):
        return [self.image(os.path.join(self.base, self.doc["images"][int(t["source"])]["uri"])) for t in self.doc.get("textures", [])]


def _opened(path):
    return path if isinstance(path, GltfFile) else GltfFile(path)


def animation_range(path, animation=0):
    """[t0, t1]: the first and the last key time of animation `animation` of a glTF file (a path or a GltfFile), in
    seconds.  Raises AnimationError when the file has no such animation."""
    src = _opened(path)
    anim = _animation(src.doc, animation)
    times = [_float_accessor(src.doc, src.buffers, int(s["input"])).reshape(-1) for s in anim["samplers"]]
    return float(min(t.min() for t in times)), float(max(t.max() for t in times))


def _slerp(q0, q1, u):
    """Shortest-arc spherical interpolation of unit quaternions (x, y, z, w) in float64, normalised."""
    d = float(np.dot(q0, q1))
    if d < 0:
        q1, d = -q1, -d
    if d > 1.0 - 1e-9:
        q = q0 + u * (q1 - q0)
    else:
        th = np.arccos(min(d, 1.0))
        q = (np.sin((1 - u) * th) * q0 + np.sin(u * th) * q1) / np.sin(th)
    return q / np.linalg.norm(q)


def sample_channel(times, values, interpolation, path, t):
    """The value of one animation sampler at time t (float32): times clamp at both ends, a key's own time returns the
    stored key value itself, and between keys LINEAR interpolates (slerp for rotations) and STEP holds the earlier key."""
    times = np.asarray(times, F).reshape(-1)
    if interpolation not in ("LINEAR", "STEP"):
        raise AnimationError(f"{interpolation} interpolation is not supported")
    t = float(t)
    if t <= float(times[0]):
        return values[0].copy()
    if t >= float(times[-1]):
        return values[-1].copy()
    k = int(np.searchsorted(times.astype(np.float64), t, side="right")) - 1  # times[k] <= t < times[k + 1]
    if float(times[k]) == t or interpolation == "STEP":
        return values[k].copy()
    u = (t - float(times[k])) / (float(times[k + 1]) - float(times[k]))
    a, b = values[k].astype(np.float64), values[k + 1].astype(np.float64)
    return (_slerp(a, b, u) if path == "rotation" else a + u * (b - a)).astype(F)


def _animated_trs(doc, buffers, animation, time):
    """{node: {"translation" | "rotation" | "scale": float32 value}} of animation `animation` at `time`."""
    anim = _animation(doc, animation)
    if doc.get("skins") or any("skin" in n for n in doc.get("nodes", [])):
        raise AnimationError("skinned meshes are not supported")
    out = {}
    for ch in anim["channels"]:
        path, node = ch["target"]["path"], ch["target"].get("node")
        smp = anim["samplers"][int(ch["sampler"])]
        interpolation = smp.get("interpolation", "LINEAR")
        if path == "weights":
            raise AnimationError("morph-target weights are not supported")
        if interpolation == "CUBICSPLINE":
            raise AnimationError("CUBICSPLINE interpolation is not supported")
        if node is None or path not in ("translation", "rotation", "scale"):
            continue
        times = _float_accessor(doc, buffers, int(smp["input"]))
        values = _float_accessor(doc, buffers, int(smp["output"]))
        out.setdefault(int(node), {})[path] = sample_channel(times, values, interpolation, path, time)
    return out


def load_gltf(path, aspect_ratio, build_bvh=True, env_map=None, add_light_triangle=None, time=None, animation=0):
    """parse_gltf_scene(path, ar) + RaytracerStaticContext (both BVH builds) -> SceneData.

    `aspect_ratio` is width/height as the CLI passes it (src/main.cpp:27).  `env_map`: image file used as the
    equirectangular environment map `Scene::bg` (what main.cpp:29-31 loads when USE_ENV_MAP is compiled in; None =
    HEAD's constant white sky).  `path` may be a GltfFile (read once, flattened many times).  `time` (seconds): the scene at that time of animation `animation`; its translation,
    rotation and scale channels replace the targeted nodes' TRS before the node transform is composed (LINEAR and
    STEP samplers; CUBICSPLINE, morph-target weights and skins raise AnimationError).  time=None ignores animations."""
    src = _opened(path)
    doc, buffers = src.doc, src.buffers
    animated = {} if time is None else _animated_trs(doc, buffers, animation, time)

    tex_images = src.textures()

    def accessor_raw(idx, dtype, comps):
        """interpret_accessor, scene.h:118-133: bufferView byteOffset only, tightly packed."""
        acc = doc["accessors"][idx]
        view = doc["bufferViews"][int(acc["bufferView"])]
        off = int(view.get("byteOffset", 0))
        count = int(acc["count"])
        buf = buffers[int(view["buffer"])]
        return buf[off:off + count * comps * np.dtype(dtype).itemsize].view(dtype).reshape(count, comps)

    def load_indices(idx):
        """load_indices, scene.h:142-181."""
        acc = doc["accessors"][idx]
        view = doc["bufferViews"][int(acc["bufferView"])]
        off = int(view.get("byteOffset", 0)) + int(acc.get("byteOffset", 0))
        ctype = int(acc["componentType"])
        if ctype not in _COMPONENT:
            raise RuntimeError("illegal scalar type")
        dt = np.dtype(_COMPONENT[ctype])
        count = int(acc["count"])
        return buffers[int(view["buffer"])][off:off + count * dt.itemsize].view(dt).astype(np.int64)

    cam = {}
    cameras = []  # every camera node, in traversal order; the reference keeps only the last perspective one (cam)
    projections = []  # the projection of each entry of `cameras`
    pos_chunks, nrm_chunks, uv_chunks, tan_chunks, mat_chunks = [], [], [], [], []
    materials = []
    mat_index = {}

    def material_id(midx):
        m = doc["materials"][midx]
        emission = np.zeros(3, F)
        if "emissiveFactor" in m:
            emission = np.array(m["emissiveFactor"], F)
        strength = m.get("extensions", {}).get("KHR_materials_emissive_strength", {}).get("emissiveStrength")
        if strength is not None:
            emission = emission * F(strength)
        rec = np.zeros((), MATERIAL_DTYPE)
        rec["color"] = (1, 1, 1, 1)
        rec["roughness"], rec["metallic"], rec["ior"] = 1.0, 1.0, 1.5
        rec["color_tex"] = rec["emissive_tex"] = rec["metallic_roughness_tex"] = rec["normal_tex"] = -1
        if "emissiveTexture" in m:
            rec["emissive_tex"] = int(m["emissiveTexture"]["index"])
        rec["emission"] = emission
        pbr = m.get("pbrMetallicRoughness")
        if pbr is not None:
            if "baseColorFactor" in pbr:
                rec["color"] = np.array(pbr["baseColorFactor"], F)
            if "baseColorTexture" in pbr:
                rec["color_tex"] = int(pbr["baseColorTexture"]["index"])
            if "metallicRoughnessTexture" in pbr:
                rec["metallic_roughness_tex"] = int(pbr["metallicRoughnessTexture"]["index"])
            rec["roughness"] = F(pbr["roughnessFactor"]) if "roughnessFactor" in pbr else F(1)
            rec["metallic"] = F(pbr["metallicFactor"]) if "metallicFactor" in pbr else F(1)
        if "normalTexture" in m:
            rec["normal_tex"] = int(m["normalTexture"]["index"])
        for t in ("color_tex", "emissive_tex", "metallic_roughness_tex", "normal_tex"):
            if rec[t] >= len(tex_images):
                raise IndexError("texture index out of range")  # res.textures.at(), scene.h:275
        key = rec.tobytes()
        if key not in mat_index:  # the reference copies the material into every Object; deduplicate here
            mat_index[key] = len(materials)
            materials.append(rec)
        return mat_index[key]

    def handle_node(node_idx, parent):
        node = doc["nodes"][node_idx]
        if node_idx in animated:
            node = {**node, **animated[node_idx]}
        rotation = node.get("rotation", [0, 0, 0, 1])
        translation = np.array(node.get("translation", [0, 0, 0]), F)
        scale = np.array(node.get("scale", [1, 1, 1]), F)
        trs = _parse_mat4(node["matrix"]) if "matrix" in node else np.eye(4, dtype=F)
        local = _mat_mul(_mat_mul(_translation(translation), _rotation(rotation)), _scale(scale))
        transform = _mat_mul(_mat_mul(parent, trs), local)
        normal_transform = _normal_matrix(transform)

        if "camera" in node:
            cdef = doc["cameras"][int(node["camera"])]

            def col_dir(v):  # norm(transform * vec4(v, 0)).xyz with vec4 length
                r = np.array([F(F(F(F(transform[i, 0] * v[0]) + F(transform[i, 1] * v[1])) + F(transform[i, 2] * v[2]))
                                + F(transform[i, 3] * F(0))) for i in range(4)], F)
                ln = np.sqrt(F(F(F(r[0] * r[0]) + F(r[1] * r[1])) + F(r[2] * r[2])) + F(r[3] * r[3]))
                return (r / ln)[:3]

        if "camera" in node and "perspective" not in cdef and "orthographic" in cdef:
            # an orthographic node joins `cameras` only: the scene camera (the reference's, which reads perspective
            # cameras alone) stays the last perspective node; fov_x is unused by the projection
            ortho = cdef["orthographic"]
            cameras.append(Camera(transform[:3, 3].copy(), col_dir(np.array([1, 0, 0], F)), col_dir(np.array([0, 1, 0], F)),
                                  col_dir(np.array([0, 0, -1], F)), F(0)))
            projections.append(Projection.orthographic(F(ortho["xmag"]), F(ortho["ymag"])))
        elif "camera" in node:
            persp = cdef["perspective"]
            fov_y = F(persp["yfov"])
            ar = F(persp["aspectRatio"]) if "aspectRatio" in persp else F(aspect_ratio)
            cam["position"] = transform[:3, 3].copy()
            cam["forward"] = col_dir(np.array([0, 0, -1], F))
            cam["up"] = col_dir(np.array([0, 1, 0], F))
            cam["right"] = col_dir(np.array([1, 0, 0], F))
            cam["fov_x"] = F(atanf(F(tanf(F(fov_y / F(2))) * ar)) * F(2))
            cameras.append(Camera(cam["position"], cam["right"], cam["up"], cam["forward"], cam["fov_x"]))
            projections.append(Projection.pinhole())

        if "mesh" in node:
            for prim in doc["meshes"][int(node["mesh"])]["primitives"]:
                mid = material_id(int(prim["material"]))
                attrs = prim["attributes"]
                coords = accessor_raw(int(attrs["POSITION"]), np.float32, 3)
                normals = accessor_raw(int(attrs["NORMAL"]), np.float32, 3) if "NORMAL" in attrs else None
                tangents = accessor_raw(int(attrs["tangent"]), np.float32, 3) if "tangent" in attrs else None
                texcoords = accessor_raw(int(attrs["TEXCOORD_0"]), np.float32, 2) if "TEXCOORD_0" in attrs else None
                indices = load_indices(int(prim["indices"]))  # required by the reference (scene.h:362)
                mode = int(prim.get("mode", 4))
                cnt = len(indices)
                if mode == 4:
                    n_t = cnt // 3
                    tri = indices[:n_t * 3].reshape(n_t, 3)
                elif mode == 5:
                    i = np.arange(2, cnt)
                    off = i & 1
                    tri = np.stack([indices[i - 2], indices[i - 1 + off], indices[i - off]], 1) if cnt > 2 \
                        else np.zeros((0, 3), np.int64)
                else:
                    continue  # the reference's switch ignores other modes (scene.h:444-458)
                if len(tri) == 0:
                    continue
                wp = _apply_points(transform, np.ascontiguousarray(coords, F))
                p = wp[tri]  # [n, 3, 3]
                if normals is not None:
                    wn = _apply_normals(normal_transform, np.ascontiguousarray(normals, F))
                    nn = wn[tri]
                else:  # obj.shape.normal(), scene.h:427-430
                    v, u = p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]
                    c = np.stack([v[:, 1] * u[:, 2] - v[:, 2] * u[:, 1], v[:, 2] * u[:, 0] - v[:, 0] * u[:, 2],
                                  v[:, 0] * u[:, 1] - v[:, 1] * u[:, 0]], 1)
                    nn = np.repeat(_normalize(c)[:, None, :], 3, axis=1)
                uv = texcoords[tri] if texcoords is not None else np.zeros((len(tri), 3, 2), F)
                tg = tangents[tri] if tangents is not None else np.tile(np.array([1, 0, 0], F), (len(tri), 3, 1))
                pos_chunks.append(p.astype(F))
                nrm_chunks.append(nn.astype(F))
                uv_chunks.append(np.asarray(uv, F))
                tan_chunks.append(np.asarray(tg, F))
                mat_chunks.append(np.full(len(tri), mid, np.uint32))
        for child in node.get("children", []):
            handle_node(int(child), transform)

    scene_idx = int(doc.get("scene", 0))
    scenes = doc.get("scenes")
    roots = scenes[scene_idx]["nodes"] if scenes and scene_idx < len(scenes) and scenes[scene_idx] is not None \
        else range(len(doc.get("nodes", [])))
    for n in roots:
        handle_node(int(n), np.eye(4, dtype=F))

    s = SceneData()
    s.cameras = cameras
    s.projections = projections
    if cam:
        s.camera_position, s.camera_right = cam["position"], cam["right"]
        s.camera_up, s.camera_forward, s.fov_x = cam["up"], cam["forward"], cam["fov_x"]
    else:  # Camera{} defaults, scene.h:60-67
        s.camera_position = np.zeros(3, F)
        s.camera_right = s.camera_up = s.camera_forward = np.zeros(3, F)
        s.fov_x = F(0)
    s.bg_color = np.ones(3, F)  # main.cpp:28 (ENV_MAP_INTENSITY)
    if pos_chunks:
        s.tri_pos = np.concatenate(pos_chunks)
        s.tri_normals = np.concatenate(nrm_chunks)
        s.tri_uv = np.concatenate(uv_chunks)
        s.tri_tangents = np.concatenate(tan_chunks)
        s.tri_material = np.concatenate(mat_chunks)
    else:
        s.tri_tangents = np.zeros((0, 3, 3), F)
    if add_light_triangle is None:
        add_light_triangle = os.environ.get("RT_ADD_LIGHT_TRIANGLE", "0") not in ("", "0")
    if add_light_triangle:
        # ADD_LIGHT_TRIANGLE (config.h:39-47, false at HEAD; scene.h:479-498): one more object after all others — the
        # triangle w + (x * right + y * up + z * forward), default material (geometry.h:604-609) with emission 10,
        # its own normal on every vertex, uv 0, tangent (1, 0, 0)
        x, y, z, w = s.camera_right.astype(F), s.camera_up.astype(F), s.camera_forward.astype(F), s.camera_position.astype(F)
        tri = np.stack([w + ((F(r[0]) * x + F(r[1]) * y) + F(r[2]) * z) for r in LIGHT_TRIANGLE_RELATIVE_POS]).astype(F)
        v, u = tri[1] - tri[0], tri[2] - tri[0]
        c = np.array([[v[1] * u[2] - v[2] * u[1], v[2] * u[0] - v[0] * u[2], v[0] * u[1] - v[1] * u[0]]], F)
        rec = np.zeros((), MATERIAL_DTYPE)
        rec["color"] = (1, 1, 1, 1)
        rec["emission"] = (LIGHT_TRIANGLE_INTENSITY,) * 3
        rec["roughness"], rec["metallic"], rec["ior"] = 1.0, 1.0, 1.5
        rec["color_tex"] = rec["emissive_tex"] = rec["metallic_roughness_tex"] = rec["normal_tex"] = -1
        key = rec.tobytes()
        if key not in mat_index:
            mat_index[key] = len(materials)
            materials.append(rec)
        empty = s.n_tris == 0
        cat = (lambda a, b: b) if empty else (lambda a, b: np.concatenate([a, b]))
        s.tri_pos = cat(s.tri_pos, tri[None])
        s.tri_normals = cat(s.tri_normals, np.repeat(_normalize(c)[:, None, :], 3, axis=1).astype(F))
        s.tri_uv = cat(s.tri_uv, np.zeros((1, 3, 2), F))
        s.tri_tangents = cat(s.tri_tangents, np.tile(np.array([1, 0, 0], F), (1, 3, 1)))
        s.tri_material = cat(s.tri_material, np.array([mat_index[key]], np.uint32))
    s.materials = np.array(materials, MATERIAL_DTYPE) if materials else np.zeros(0, MATERIAL_DTYPE)
    if env_map is not None:
        env = src.image(env_map)
        if env.shape[0] * env.shape[1] > 1 or not (env[0, 0, :3] == 255).all():  # 1x1 white = HEAD's constant sky
            tex_images = tex_images + [env]
            s.env_texture = len(tex_images)
    tex = np.zeros(len(tex_images), TEXTURE_DTYPE)
    blobs, off = [], 0
    for i, im in enumerate(tex_images):
        tex[i] = (im.shape[1], im.shape[0], off)
        blobs.append(im.reshape(-1))
        off += im.size
    s.textures = tex
    s.texels = np.concatenate(blobs) if blobs else np.zeros(0, np.uint8)
    if build_bvh:
        build_bvhs(s)
    return s


def build_bvhs(s):
    """RaytracerStaticContext, raytracer.h:440-447: BVH over all objects + BVH over emission != 0."""
    s.scene_bvh = host.build_bvh(s.tri_pos)
    return build_light_bvh(s)


def build_light_bvh(s):
    """The BVH over emission != 0 alone (raytracer.h:444-447): what an update of moved geometry passes."""
    if s.n_tris:
        em = s.materials["emission"][s.tri_material]
        s.light_bvh = host.build_bvh(s.tri_pos, select=(em != 0).any(axis=1))
    else:
        s.light_bvh = host.build_bvh(s.tri_pos)
    return s
