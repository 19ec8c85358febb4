"""ctypes mirror of include/rt_gpu.h and the RTSC container (host/rt_host.cpp).

`SceneData` owns the flattened scene as numpy arrays (the host-side equivalent of the reference's
`Scene` + `RaytracerStaticContext`, src/scene.h:74-90, src/raytracer.h:434-455) and hands out a
ctypes `rt_scene_desc` whose pointers alias those arrays.
"""
import ctypes as C
import os

import numpy as np

RT_GPU_ABI_VERSION = 1
RT_NO_CHILD = 0xFFFFFFFF

RT_MODE_BEAUTY = 0
RT_MODE_PRIMARY_IDS = 1
RT_FLAG_ACCUMULATE = 1

STATUS = {
    0: "RT_OK", -1: "RT_ERR_INVALID_ARG", -2: "RT_ERR_NO_DEVICE", -3: "RT_ERR_CUDA", -4: "RT_ERR_NO_SCENE",
    -5: "RT_ERR_NO_RENDER", -6: "RT_ERR_NCCL", -7: "RT_ERR_BAD_SCENE", -8: "RT_ERR_OOM",
}

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT_DIR = os.path.dirname(PKG_DIR)

# numpy dtypes of the POD records (layout == the C structs)
NODE_DTYPE = np.dtype([("bmin", "<f4", 3), ("bmax", "<f4", 3), ("left_child", "<u4"), ("right_child", "<u4"),
                       ("obj_begin", "<u4"), ("obj_end", "<u4")])
MATERIAL_DTYPE = np.dtype([("color", "<f4", 4), ("emission", "<f4", 3), ("roughness", "<f4"), ("metallic", "<f4"),
                           ("ior", "<f4"), ("color_tex", "<i4"), ("emissive_tex", "<i4"),
                           ("metallic_roughness_tex", "<i4"), ("normal_tex", "<i4")])
TEXTURE_DTYPE = np.dtype([("width", "<u4"), ("height", "<u4"), ("offset", "<u8")])
assert NODE_DTYPE.itemsize == 40 and MATERIAL_DTYPE.itemsize == 56 and TEXTURE_DTYPE.itemsize == 16

RTSC_HEADER = np.dtype([
    ("magic", "S8"), ("abi_version", "<u4"), ("n_tris", "<u4"),
    ("cam_position", "<f4", 3), ("cam_right", "<f4", 3), ("cam_up", "<f4", 3), ("cam_forward", "<f4", 3),
    ("fov_x", "<f4"), ("bg_color", "<f4", 3), ("eps", "<f4"), ("min_roughness", "<f4"), ("vndf_factor", "<f4"),
    ("ray_depth", "<u4"), ("n_materials", "<u4"), ("n_textures", "<u4"), ("has_tangents", "<u4"), ("env_texture", "<u4"),
    ("texel_bytes", "<u8"),
    ("scene_n_nodes", "<u4"), ("scene_root", "<u4"), ("scene_n_objects", "<u4"),
    ("light_n_nodes", "<u4"), ("light_root", "<u4"), ("light_n_objects", "<u4"),
])
assert RTSC_HEADER.itemsize == 144


class rt_bvh_node(C.Structure):
    _fields_ = [("bmin", C.c_float * 3), ("bmax", C.c_float * 3), ("left_child", C.c_uint32),
                ("right_child", C.c_uint32), ("obj_begin", C.c_uint32), ("obj_end", C.c_uint32)]


class rt_bvh_desc(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("root", C.c_uint32), ("n_objects", C.c_uint32), ("_pad", C.c_uint32),
                ("nodes", C.c_void_p), ("objects", C.c_void_p)]


class rt_camera(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("right", C.c_float * 3), ("up", C.c_float * 3),
                ("forward", C.c_float * 3), ("fov_x", C.c_float)]


class rt_views(C.Structure):
    _fields_ = [("n_views", C.c_uint32), ("view_base", C.c_uint32), ("cameras", C.POINTER(rt_camera))]


RT_PROJ_PINHOLE, RT_PROJ_THIN_LENS, RT_PROJ_ORTHOGRAPHIC, RT_PROJ_EQUIRECT = 0, 1, 2, 3


class rt_projection(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("aperture_radius", C.c_float), ("focus_distance", C.c_float), ("half_width", C.c_float),
                ("half_height", C.c_float)]


class Projection:
    """How a view maps pixels to rays (rt_projection, include/rt_gpu.h): Projection.pinhole(), thin_lens(aperture_radius,
    focus_distance), orthographic(half_width, half_height) (glTF xmag / ymag) or equirect().  Fields a kind does not use
    are 0.  Two projections are equal when kind and every value are equal bit for bit."""

    __slots__ = ("kind", "aperture_radius", "focus_distance", "half_width", "half_height")
    NAMES = {RT_PROJ_PINHOLE: "pinhole", RT_PROJ_THIN_LENS: "thin_lens", RT_PROJ_ORTHOGRAPHIC: "ortho", RT_PROJ_EQUIRECT: "equirect"}

    def __init__(self, kind=RT_PROJ_PINHOLE, aperture_radius=0.0, focus_distance=0.0, half_width=0.0, half_height=0.0):
        self.kind = int(kind)
        self.aperture_radius, self.focus_distance = np.float32(aperture_radius), np.float32(focus_distance)
        self.half_width, self.half_height = np.float32(half_width), np.float32(half_height)

    @classmethod
    def pinhole(cls):
        return cls(RT_PROJ_PINHOLE)

    @classmethod
    def thin_lens(cls, aperture_radius, focus_distance):
        return cls(RT_PROJ_THIN_LENS, aperture_radius=aperture_radius, focus_distance=focus_distance)

    @classmethod
    def orthographic(cls, half_width, half_height):
        return cls(RT_PROJ_ORTHOGRAPHIC, half_width=half_width, half_height=half_height)

    @classmethod
    def equirect(cls):
        return cls(RT_PROJ_EQUIRECT)

    @classmethod
    def parse(cls, text):
        """The CLI form: 'pinhole', 'thin_lens:<aperture>:<focus>', 'ortho:<half_w>:<half_h>' or 'equirect'."""
        name, *args = text.split(":")
        makers = {"pinhole": (cls.pinhole, 0), "thin_lens": (cls.thin_lens, 2), "ortho": (cls.orthographic, 2), "equirect": (cls.equirect, 0)}
        if name not in makers or len(args) != makers[name][1]:
            raise ValueError(f"projection {text!r}: expected pinhole, thin_lens:<aperture>:<focus>, ortho:<half_w>:<half_h> or equirect")
        return makers[name][0](*(float(a) for a in args))

    def to_c(self):
        return rt_projection(self.kind, float(self.aperture_radius), float(self.focus_distance), float(self.half_width),
                             float(self.half_height))

    def _bits(self):
        return (self.kind, np.array([self.aperture_radius, self.focus_distance, self.half_width, self.half_height],
                                    np.float32).view(np.uint32).tolist())

    def __eq__(self, other):
        return isinstance(other, Projection) and self._bits() == other._bits()

    __hash__ = None

    def __repr__(self):
        return (f"Projection({self.NAMES.get(self.kind, self.kind)}, aperture_radius={float(self.aperture_radius)!r}, "
                f"focus_distance={float(self.focus_distance)!r}, half_width={float(self.half_width)!r}, "
                f"half_height={float(self.half_height)!r})")


class Camera:
    """A camera of a scene (rt_camera): position, the right / up / forward axes and the horizontal field of view fov_x
    in radians, all float32.  Two cameras are equal when every value is equal bit for bit."""

    __slots__ = ("position", "right", "up", "forward", "fov_x")

    def __init__(self, position, right, up, forward, fov_x):
        self.position = np.array(position, np.float32).reshape(3)
        self.right = np.array(right, np.float32).reshape(3)
        self.up = np.array(up, np.float32).reshape(3)
        self.forward = np.array(forward, np.float32).reshape(3)
        self.fov_x = np.float32(fov_x)

    def to_c(self):
        c = rt_camera()
        for k in range(3):
            c.position[k], c.right[k] = float(self.position[k]), float(self.right[k])
            c.up[k], c.forward[k] = float(self.up[k]), float(self.forward[k])
        c.fov_x = float(self.fov_x)
        return c

    def _bits(self):
        return np.concatenate([self.position, self.right, self.up, self.forward, [self.fov_x]]).astype(np.float32).view(np.uint32)

    def __eq__(self, other):
        return isinstance(other, Camera) and np.array_equal(self._bits(), other._bits())

    __hash__ = None

    def __repr__(self):
        return (f"Camera(position={self.position.tolist()}, right={self.right.tolist()}, up={self.up.tolist()}, "
                f"forward={self.forward.tolist()}, fov_x={float(self.fov_x)!r})")


class rt_scene_desc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32), ("n_tris", C.c_uint32), ("camera", rt_camera), ("bg_color", C.c_float * 3),
        ("eps", C.c_float), ("min_roughness", C.c_float), ("vndf_factor", C.c_float), ("ray_depth", C.c_uint32),
        ("n_materials", C.c_uint32), ("n_textures", C.c_uint32), ("flags", C.c_uint32), ("env_texture", C.c_uint32),
        ("texel_bytes", C.c_uint64),
        ("tri_pos", C.c_void_p), ("tri_normals", C.c_void_p), ("tri_uv", C.c_void_p), ("tri_tangents", C.c_void_p),
        ("tri_material", C.c_void_p), ("materials", C.c_void_p), ("textures", C.c_void_p), ("texels", C.c_void_p),
        ("scene_bvh", rt_bvh_desc), ("light_bvh", rt_bvh_desc),
    ]


class rt_render_params(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("samples", C.c_uint32), ("sample_begin", C.c_uint32),
                ("sample_end", C.c_uint32), ("mode", C.c_uint32), ("seed", C.c_uint64),
                ("max_paths_in_flight", C.c_uint32), ("flags", C.c_uint32), ("pixel_begin", C.c_uint32),
                ("pixel_end", C.c_uint32)]


class rt_adaptive_params(C.Structure):
    _fields_ = [("min_samples", C.c_uint32), ("step_samples", C.c_uint32), ("rel_error", C.c_float), ("abs_floor", C.c_float)]


class rt_stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("extension_rays", C.c_uint64), ("light_pdf_rays", C.c_uint64),
                ("shades", C.c_uint64), ("render_ms", C.c_double), ("reduce_ms", C.c_double),
                ("kernel_ms", C.c_double * 8), ("kernel_launches", C.c_uint64)]

    def as_dict(self):
        return {"samples": self.samples, "extension_rays": self.extension_rays,
                "light_pdf_rays": self.light_pdf_rays, "shades": self.shades, "render_ms": self.render_ms,
                "reduce_ms": self.reduce_ms, "kernel_ms": list(self.kernel_ms),
                "kernel_launches": self.kernel_launches}


class rt_bvh_build(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("root", C.c_uint32), ("n_objects", C.c_uint32), ("_pad", C.c_uint32),
                ("nodes", C.c_void_p), ("objects", C.c_void_p)]


def _ptr(a):
    return a.ctypes.data if a is not None and a.size else None


class BvhData:
    def __init__(self, nodes, objects, root):
        self.nodes = np.ascontiguousarray(nodes, dtype=NODE_DTYPE)
        self.objects = np.ascontiguousarray(objects, dtype=np.uint32)
        self.root = int(root) if len(self.objects) else RT_NO_CHILD

    def desc(self):
        d = rt_bvh_desc()
        d.n_nodes = len(self.nodes)
        d.root = self.root
        d.n_objects = len(self.objects)
        d.nodes = _ptr(self.nodes)
        d.objects = _ptr(self.objects)
        return d


class SceneData:
    """Flattened scene in host memory (numpy). Field meaning: include/rt_gpu.h `rt_scene_desc`."""

    def __init__(self):
        self.camera_position = np.zeros(3, np.float32)
        self.camera_right = np.array([1, 0, 0], np.float32)
        self.camera_up = np.array([0, 1, 0], np.float32)
        self.camera_forward = np.array([0, 0, -1], np.float32)
        self.fov_x = np.float32(1.0)
        self.bg_color = np.ones(3, np.float32)            # main.cpp:28
        self.eps = np.float32(1e-4)                       # config.h:15
        self.min_roughness = np.float32(0.04)             # config.h:20
        self.vndf_factor = np.float32(1.0) / np.float32(3)  # config.h:26
        self.ray_depth = 8                                # config.h:17
        self.env_texture = 0                              # 0 = constant sky; k + 1 = textures[k] is Scene::bg
        self.tri_pos = np.zeros((0, 3, 3), np.float32)
        self.tri_normals = np.zeros((0, 3, 3), np.float32)
        self.tri_uv = np.zeros((0, 3, 2), np.float32)
        self.tri_tangents = None
        self.tri_material = np.zeros(0, np.uint32)
        self.materials = np.zeros(0, MATERIAL_DTYPE)
        self.textures = np.zeros(0, TEXTURE_DTYPE)
        self.texels = np.zeros(0, np.uint8)
        self.scene_bvh = BvhData(np.zeros(0, NODE_DTYPE), np.zeros(0, np.uint32), RT_NO_CHILD)
        self.light_bvh = BvhData(np.zeros(0, NODE_DTYPE), np.zeros(0, np.uint32), RT_NO_CHILD)
        self.cameras = []  # every camera node of the source glTF in traversal order (gltf.load_gltf); the scene's own
                           # camera is the last perspective one
        self.projections = []  # the Projection of each entry of `cameras`

    def camera(self):
        """The scene's own camera (the one rt_gpu_render uses) as a Camera."""
        return Camera(self.camera_position, self.camera_right, self.camera_up, self.camera_forward, self.fov_x)

    @property
    def n_tris(self):
        return int(self.tri_pos.shape[0])

    def _normalise(self):
        n = self.n_tris
        self.tri_pos = np.ascontiguousarray(self.tri_pos, np.float32).reshape(n, 3, 3)
        self.tri_normals = np.ascontiguousarray(self.tri_normals, np.float32).reshape(n, 3, 3)
        self.tri_uv = np.ascontiguousarray(self.tri_uv, np.float32).reshape(n, 3, 2)
        if self.tri_tangents is not None:
            self.tri_tangents = np.ascontiguousarray(self.tri_tangents, np.float32).reshape(n, 3, 3)
        self.tri_material = np.ascontiguousarray(self.tri_material, np.uint32)
        self.materials = np.ascontiguousarray(self.materials, MATERIAL_DTYPE)
        self.textures = np.ascontiguousarray(self.textures, TEXTURE_DTYPE)
        self.texels = np.ascontiguousarray(self.texels, np.uint8)

    def without_scene_bvh(self):
        """Shallow copy that passes no scene BVH (rt_gpu.h: scene_bvh.n_nodes == 0 -> the library builds it)."""
        import copy

        s = copy.copy(self)
        s.scene_bvh = BvhData(np.zeros(0, NODE_DTYPE), np.zeros(0, np.uint32), RT_NO_CHILD)
        return s

    def desc(self):
        """ctypes rt_scene_desc aliasing this object's arrays (keep `self` alive while it is used)."""
        self._normalise()
        d = rt_scene_desc()
        d.abi_version = RT_GPU_ABI_VERSION
        d.n_tris = self.n_tris
        for k in range(3):
            d.camera.position[k] = float(self.camera_position[k])
            d.camera.right[k] = float(self.camera_right[k])
            d.camera.up[k] = float(self.camera_up[k])
            d.camera.forward[k] = float(self.camera_forward[k])
            d.bg_color[k] = float(self.bg_color[k])
        d.camera.fov_x = float(self.fov_x)
        d.eps = float(self.eps)
        d.min_roughness = float(self.min_roughness)
        d.vndf_factor = float(self.vndf_factor)
        d.ray_depth = int(self.ray_depth)
        d.n_materials = len(self.materials)
        d.n_textures = len(self.textures)
        d.env_texture = int(self.env_texture)
        d.texel_bytes = int(self.texels.size)
        d.tri_pos = _ptr(self.tri_pos)
        d.tri_normals = _ptr(self.tri_normals)
        d.tri_uv = _ptr(self.tri_uv)
        d.tri_tangents = _ptr(self.tri_tangents)
        d.tri_material = _ptr(self.tri_material)
        d.materials = _ptr(self.materials)
        d.textures = _ptr(self.textures)
        d.texels = _ptr(self.texels)
        d.scene_bvh = self.scene_bvh.desc()
        d.light_bvh = self.light_bvh.desc()
        d._owner = self
        return d

    # ---- RTSC container (same bytes as rt_scene_save / rt_scene_load) ------------------------------
    def _sections(self):
        self._normalise()
        return [self.tri_pos, self.tri_normals, self.tri_uv, self.tri_tangents, self.tri_material, self.materials,
                self.textures, self.texels, self.scene_bvh.nodes, self.scene_bvh.objects, self.light_bvh.nodes,
                self.light_bvh.objects]

    def save(self, path):
        h = np.zeros(1, RTSC_HEADER)
        h["magic"] = b"RTSC0001"
        h["abi_version"] = RT_GPU_ABI_VERSION
        h["n_tris"] = self.n_tris
        h["cam_position"], h["cam_right"] = self.camera_position, self.camera_right
        h["cam_up"], h["cam_forward"] = self.camera_up, self.camera_forward
        h["fov_x"], h["bg_color"] = self.fov_x, self.bg_color
        h["eps"], h["min_roughness"], h["vndf_factor"] = self.eps, self.min_roughness, self.vndf_factor
        h["ray_depth"] = self.ray_depth
        h["n_materials"], h["n_textures"] = len(self.materials), len(self.textures)
        h["has_tangents"] = 0 if self.tri_tangents is None else 1
        h["env_texture"] = self.env_texture
        h["texel_bytes"] = self.texels.size
        h["scene_n_nodes"], h["scene_root"] = len(self.scene_bvh.nodes), self.scene_bvh.root
        h["scene_n_objects"] = len(self.scene_bvh.objects)
        h["light_n_nodes"], h["light_root"] = len(self.light_bvh.nodes), self.light_bvh.root
        h["light_n_objects"] = len(self.light_bvh.objects)
        with open(path, "wb") as f:
            f.write(h.tobytes())
            for sec in self._sections():
                b = b"" if sec is None else sec.tobytes()
                f.write(b)
                f.write(b"\0" * (-len(b) % 16))

    @staticmethod
    def load(path):
        raw = np.fromfile(path, np.uint8)
        h = raw[:RTSC_HEADER.itemsize].view(RTSC_HEADER)[0]
        if bytes(h["magic"]) != b"RTSC0001":
            raise ValueError(f"{path}: not an RTSC file")
        s = SceneData()
        n = int(h["n_tris"])
        s.camera_position, s.camera_right = h["cam_position"].copy(), h["cam_right"].copy()
        s.camera_up, s.camera_forward = h["cam_up"].copy(), h["cam_forward"].copy()
        s.fov_x, s.bg_color = np.float32(h["fov_x"]), h["bg_color"].copy()
        s.eps, s.min_roughness = np.float32(h["eps"]), np.float32(h["min_roughness"])
        s.vndf_factor, s.ray_depth = np.float32(h["vndf_factor"]), int(h["ray_depth"])
        s.env_texture = int(h["env_texture"])
        off = [RTSC_HEADER.itemsize]

        def take(dtype, count):
            dt = np.dtype(dtype)
            nbytes = dt.itemsize * count
            a = raw[off[0]:off[0] + nbytes].view(dt).copy()
            off[0] += nbytes + (-nbytes % 16)
            return a

        s.tri_pos = take("<f4", n * 9).reshape(n, 3, 3)
        s.tri_normals = take("<f4", n * 9).reshape(n, 3, 3)
        s.tri_uv = take("<f4", n * 6).reshape(n, 3, 2)
        tang = take("<f4", n * 9 if h["has_tangents"] else 0)
        s.tri_tangents = tang.reshape(n, 3, 3) if h["has_tangents"] else None
        s.tri_material = take("<u4", n)
        s.materials = take(MATERIAL_DTYPE, int(h["n_materials"]))
        s.textures = take(TEXTURE_DTYPE, int(h["n_textures"]))
        s.texels = take(np.uint8, int(h["texel_bytes"]))
        nodes = take(NODE_DTYPE, int(h["scene_n_nodes"]))
        objs = take("<u4", int(h["scene_n_objects"]))
        s.scene_bvh = BvhData(nodes, objs, int(h["scene_root"]))
        nodes = take(NODE_DTYPE, int(h["light_n_nodes"]))
        objs = take("<u4", int(h["light_n_objects"]))
        s.light_bvh = BvhData(nodes, objs, int(h["light_root"]))
        return s


def load_library(path, what):
    """dlopen an in-tree shared library; fail loudly (there is no fallback for a missing build)."""
    if not os.path.exists(path):
        raise RuntimeError(f"{what} not built: {path} is missing. Run `python -c 'import __graft_entry__ as g; "
                           f"g.build()'` at the repository root (needs nvcc / g++).")
    return C.CDLL(path)
