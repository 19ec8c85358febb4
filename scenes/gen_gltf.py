#!/usr/bin/env python3
"""Deterministic synthetic glTF scenes (the reference ships none: sample_data/.gitignore:1-2).

Every scene obeys the constraints of the reference loader (src/scene.h:183-501):
external .bin buffers, one tightly packed bufferView per accessor (accessor
byteOffset / byteStride are ignored there, scene.h:118-133), every primitive has
`material` and `indices` (scene.h:261,362), a camera node exists (scene.h:234),
images are files stb_image can decode (PPM / PNG).

Scenes
  tiny         7 triangles, Cornell-like: floor, back wall, emissive triangle, metallic quad
  small        scaled-down corridor (~2.7k triangles), env lit
  small_lights same + 32 emissive triangles
  small_manylights  same with the four panels cut into 12 x 12 quads: 1152 emissive triangles (a light BVH several levels deep)
  big          "Sponza-scale" corridor, 260 160 triangles (SURVEY.md 8(d)), env lit
  big_lights   same + 32 emissive triangles = 260 192
  texmaps      texall with every roughness >= 0.35 (well-conditioned: held to the tight path-by-path bound)
  texall       every loader / material feature: node hierarchy (matrix + TRS, non-uniform
               scale), u8/u16/u32 indices, triangle strip, missing normals, base-colour
               texture with alpha (PNG), normal map, metallic-roughness map, emissive map,
               KHR_materials_emissive_strength, 1x1 texture

usage: gen_gltf.py <scene> <out_dir>     -> <out_dir>/<scene>.gltf (+ .bin, textures)
"""
import json
import os
import sys

import numpy as np

FLOAT = 5126
U8, U16, U32 = 5121, 5123, 5125


class GltfBuilder:
    def __init__(self, name):
        self.name = name
        self.blob = bytearray()
        self.views = []
        self.accessors = []
        self.meshes = []
        self.nodes = []
        self.materials = []
        self.textures = []
        self.images = []
        self.cameras = []
        self.scene_nodes = []
        self.files = {}
        self.extensions_used = set()
        self.animations = []

    def _view(self, data: bytes):
        while len(self.blob) % 4:
            self.blob.append(0)
        off = len(self.blob)
        self.blob += data
        self.views.append({"buffer": 0, "byteOffset": off, "byteLength": len(data)})
        return len(self.views) - 1

    def accessor(self, arr, comp, typ):
        arr = np.ascontiguousarray(arr)
        view = self._view(arr.tobytes())
        count = arr.shape[0]
        acc = {"bufferView": view, "componentType": comp, "count": int(count), "type": typ}
        if typ == "VEC3" and comp == FLOAT:
            acc["min"] = [float(v) for v in arr.min(axis=0)]
            acc["max"] = [float(v) for v in arr.max(axis=0)]
        self.accessors.append(acc)
        return len(self.accessors) - 1

    def primitive(self, pos, idx, material, normals=None, uv=None, mode=None, index_type=U32):
        attrs = {"POSITION": self.accessor(pos.astype(np.float32), FLOAT, "VEC3")}
        if normals is not None:
            attrs["NORMAL"] = self.accessor(normals.astype(np.float32), FLOAT, "VEC3")
        if uv is not None:
            attrs["TEXCOORD_0"] = self.accessor(uv.astype(np.float32), FLOAT, "VEC2")
        dt = {U8: np.uint8, U16: np.uint16, U32: np.uint32}[index_type]
        prim = {
            "attributes": attrs,
            "indices": self.accessor(np.asarray(idx).reshape(-1).astype(dt), index_type, "SCALAR"),
            "material": material,
        }
        if mode is not None:
            prim["mode"] = mode
        return prim

    def mesh(self, primitives):
        self.meshes.append({"primitives": primitives})
        return len(self.meshes) - 1

    def node(self, root=True, **kw):
        self.nodes.append(kw)
        i = len(self.nodes) - 1
        if root:
            self.scene_nodes.append(i)
        return i

    def material(self, **kw):
        self.materials.append(kw)
        return len(self.materials) - 1

    def texture(self, filename, data: bytes):
        self.files[filename] = data
        self.images.append({"uri": filename})
        self.textures.append({"source": len(self.images) - 1})
        return len(self.textures) - 1

    def camera(self, yfov, aspect=None, **node_kw):
        persp = {"yfov": yfov, "znear": 0.01}
        if aspect is not None:
            persp["aspectRatio"] = aspect
        self.cameras.append({"type": "perspective", "perspective": persp})
        return self.node(camera=len(self.cameras) - 1, **node_kw)

    def animation(self, channels, name=None):
        """One glTF animation from channels (node, path, key times, key values, interpolation); path is "translation",
        "rotation", "scale" or "weights".  Returns its index."""
        samplers, chans = [], []
        comps = {"translation": 3, "rotation": 4, "scale": 3, "weights": 1}
        for node, path, times, values, interp in channels:
            t = np.asarray(times, np.float32).reshape(-1)
            inp = self.accessor(t, FLOAT, "SCALAR")
            self.accessors[inp]["min"], self.accessors[inp]["max"] = [float(t.min())], [float(t.max())]
            v = np.asarray(values, np.float32).reshape(-1, comps[path])
            out = self.accessor(v if comps[path] > 1 else v.reshape(-1), FLOAT, {1: "SCALAR", 3: "VEC3", 4: "VEC4"}[comps[path]])
            samplers.append({"input": inp, "output": out, "interpolation": interp})
            chans.append({"sampler": len(samplers) - 1, "target": {"node": node, "path": path}})
        anim = {"samplers": samplers, "channels": chans}
        if name is not None:
            anim["name"] = name
        self.animations.append(anim)
        return len(self.animations) - 1

    def write(self, out_dir):
        os.makedirs(out_dir, exist_ok=True)
        binname = self.name + ".bin"
        doc = {
            "asset": {"version": "2.0", "generator": "b200-pathtracer gen_gltf.py"},
            "scene": 0,
            "scenes": [{"nodes": self.scene_nodes}],
            "nodes": self.nodes,
            "meshes": self.meshes,
            "materials": self.materials,
            "cameras": self.cameras,
            "accessors": self.accessors,
            "bufferViews": self.views,
            "buffers": [{"uri": binname, "byteLength": len(self.blob)}],
            # the reference iterates scene_struct["textures"] unconditionally (scene.h:204)
            "textures": self.textures,
            "images": self.images,
        }
        if self.extensions_used:
            doc["extensionsUsed"] = sorted(self.extensions_used)
        if self.animations:
            doc["animations"] = self.animations
        with open(os.path.join(out_dir, binname), "wb") as f:
            f.write(bytes(self.blob))
        for fn, data in self.files.items():
            with open(os.path.join(out_dir, fn), "wb") as f:
                f.write(data)
        path = os.path.join(out_dir, self.name + ".gltf")
        with open(path, "w") as f:
            json.dump(doc, f)
        return path


def ppm_bytes(rgb):
    h, w, _ = rgb.shape
    return b"P6\n%d %d\n255\n" % (w, h) + np.ascontiguousarray(rgb, dtype=np.uint8).tobytes()


def png_bytes(rgba):
    """Minimal PNG writer (zlib only), 8-bit RGB or RGBA."""
    import struct
    import zlib

    h, w, c = rgba.shape
    ctype = {3: 2, 4: 6}[c]
    raw = b"".join(b"\x00" + np.ascontiguousarray(rgba[y], dtype=np.uint8).tobytes() for y in range(h))

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    return (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, ctype, 0, 0, 0))
            + chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))


def checker_texture(rng, size=512, cells=16):
    y, x = np.mgrid[0:size, 0:size]
    chk = ((x // (size // cells) + y // (size // cells)) & 1).astype(np.float32)
    base = 0.35 + 0.45 * chk
    noise = rng.normal(0.0, 0.06, (size, size, 3)).astype(np.float32)
    tint = np.array([1.0, 0.92, 0.8], np.float32)
    img = np.clip((base[..., None] * tint + noise) * 255.0, 0, 255).astype(np.uint8)
    return img


def grid(nu, nv, fn):
    """(nu x nv) quads; fn(u, v) -> (P[...,3]) with u,v in [0,1]. Returns pos, normals, uv, tri indices."""
    u = np.linspace(0.0, 1.0, nu + 1)
    v = np.linspace(0.0, 1.0, nv + 1)
    uu, vv = np.meshgrid(u, v, indexing="ij")
    P = fn(uu, vv).astype(np.float64)
    du = np.gradient(P, axis=0)
    dv = np.gradient(P, axis=1)
    N = np.cross(du, dv)
    N /= np.maximum(np.linalg.norm(N, axis=-1, keepdims=True), 1e-20)
    i = np.arange(nu)[:, None] * (nv + 1) + np.arange(nv)[None, :]
    a, b, c, d = i, i + (nv + 1), i + (nv + 1) + 1, i + 1
    tris = np.stack([np.stack([a, b, c], -1), np.stack([a, c, d], -1)], 2).reshape(-1, 3)
    uv = np.stack([uu, vv], -1)
    return P.reshape(-1, 3), N.reshape(-1, 3), uv.reshape(-1, 2), tris


def corridor(name, scale, lights, light_res=2):
    """Corridor 16 x 60 x 12 m open to the sky. scale=1 -> 260 160 triangles.  light_res: quads per side of each of the
    four emissive panels (2 -> 8 triangles per panel)."""
    rng = np.random.default_rng(260000)
    g = GltfBuilder(name)
    W, L, H = 16.0, 60.0, 12.0
    s = lambda n: max(2, int(round(n * scale)))

    tex = g.texture(name + "_base.ppm", ppm_bytes(checker_texture(rng, 512 if scale >= 1.0 else 128)))
    m_floor = g.material(pbrMetallicRoughness={"baseColorTexture": {"index": tex}, "metallicFactor": 0.0,
                                               "roughnessFactor": 0.9})
    m_wall = g.material(pbrMetallicRoughness={"baseColorFactor": [0.9, 0.8, 0.7, 1.0],
                                              "baseColorTexture": {"index": tex}, "metallicFactor": 0.0,
                                              "roughnessFactor": 0.7})
    m_end = g.material(pbrMetallicRoughness={"baseColorFactor": [0.7, 0.7, 0.75, 1.0], "metallicFactor": 0.0,
                                             "roughnessFactor": 0.5})
    m_col = g.material(pbrMetallicRoughness={"baseColorFactor": [0.95, 0.8, 0.5, 1.0], "metallicFactor": 1.0,
                                             "roughnessFactor": 0.3})
    g.extensions_used.add("KHR_materials_emissive_strength")
    m_light = g.material(pbrMetallicRoughness={"baseColorFactor": [0.0, 0.0, 0.0, 1.0], "metallicFactor": 0.0,
                                               "roughnessFactor": 1.0},
                         emissiveFactor=[1.0, 0.9, 0.8],
                         extensions={"KHR_materials_emissive_strength": {"emissiveStrength": 15.0}})

    prims = []

    def add(P, N, UV, T, mat, uvscale=4.0):
        prims.append(g.primitive(P, T, mat, normals=N, uv=UV * uvscale))

    # floor: y = 1 cm bump (sinus + noise)
    nu, nv = s(140), s(280)
    nz = rng.normal(0.0, 0.3, (nu + 1, nv + 1))

    def floor(u, v):
        x = (u - 0.5) * W
        z = v * L
        y = 0.01 * (np.sin(2.0 * x) * np.sin(2.0 * z) + nz)
        return np.stack([x, y, z], -1)

    P, N, UV, T = grid(nu, nv, floor)
    add(P, N, UV * np.array([4.0, 15.0]), T[:, [0, 2, 1]], m_floor, 1.0)

    # side walls: 5 cm bump
    for side in (-1.0, 1.0):
        nu, nv = s(220), s(100)
        nz = rng.normal(0.0, 0.3, (nu + 1, nv + 1))

        def wall(u, v, side=side, nz=nz):
            z = u * L
            y = v * H
            x = side * (W / 2) + 0.05 * (np.sin(1.5 * z) * np.sin(2.0 * y) + nz)
            return np.stack([x, y, z], -1)

        P, N, UV, T = grid(nu, nv, wall)
        add(P, N, UV * np.array([15.0, 3.0]), T if side < 0 else T[:, [0, 2, 1]], m_wall, 1.0)

    # end walls
    for zpos in (0.0, L):
        nu, nv = s(100), s(100)

        def endw(u, v, zpos=zpos):
            x = (u - 0.5) * W
            y = v * H
            z = np.full_like(x, zpos) + 0.02 * np.sin(3.0 * x) * np.sin(3.0 * y)
            return np.stack([x, y, z], -1)

        P, N, UV, T = grid(nu, nv, endw)
        add(P, N, UV, T if zpos > 0 else T[:, [0, 2, 1]], m_end)

    # 20 fluted columns
    for k in range(20):
        cx = -5.5 if k % 2 == 0 else 5.5
        cz = 3.0 + 6.0 * (k // 2)
        nu, nv = s(32), s(42)

        def col(u, v, cx=cx, cz=cz):
            th = 2.0 * np.pi * u
            r = 0.6 + 0.05 * np.cos(8.0 * th) - 0.1 * v
            return np.stack([cx + r * np.cos(th), v * H, cz + r * np.sin(th)], -1)

        P, N, UV, T = grid(nu, nv, col)
        add(P, N, UV, T[:, [0, 2, 1]], m_col)

    if lights:
        for k in range(4):
            cz = 10.0 + 13.0 * k

            def panel(u, v, cz=cz):
                return np.stack([(u - 0.5) * 2.0, np.full_like(u, 8.0), cz + (v - 0.5) * 2.0], -1)

            P, N, UV, T = grid(light_res, light_res, panel)
            add(P, N, UV, T, m_light)

    g.node(mesh=g.mesh(prims))
    g.camera(1.0, translation=[0.0, 2.0, L - 2.0])
    return g


def tiny():
    g = GltfBuilder("tiny")
    m_floor = g.material(pbrMetallicRoughness={"baseColorFactor": [0.8, 0.8, 0.8, 1.0], "metallicFactor": 0.0,
                                               "roughnessFactor": 0.8})
    m_back = g.material(pbrMetallicRoughness={"baseColorFactor": [0.8, 0.3, 0.25, 1.0], "metallicFactor": 0.0,
                                              "roughnessFactor": 0.6})
    m_metal = g.material(pbrMetallicRoughness={"baseColorFactor": [0.9, 0.85, 0.6, 1.0], "metallicFactor": 1.0,
                                               "roughnessFactor": 0.25})
    m_light = g.material(pbrMetallicRoughness={"baseColorFactor": [0.0, 0.0, 0.0, 1.0], "metallicFactor": 0.0},
                         emissiveFactor=[6.0, 5.0, 4.0])
    f32 = np.float32
    floor = np.array([[-3, 0, -6], [3, 0, -6], [3, 0, 1], [-3, 0, 1]], f32)
    back = np.array([[-3, 0, -6], [3, 0, -6], [3, 4, -6], [-3, 4, -6]], f32)
    quad = np.array([[0.4, 0.0, -4.5], [2.2, 0.0, -3.6], [2.2, 1.8, -3.6], [0.4, 1.8, -4.5]], f32)
    light = np.array([[-1.6, 3.2, -4.5], [-0.2, 3.4, -4.0], [-1.2, 3.0, -3.0]], f32)
    up = np.tile(np.array([[0, 1, 0]], f32), (4, 1))
    fw = np.tile(np.array([[0, 0, 1]], f32), (4, 1))
    prims = [
        g.primitive(floor, [0, 2, 1, 0, 3, 2], m_floor, normals=up, index_type=U16),
        g.primitive(back, [0, 1, 2, 0, 2, 3], m_back, normals=fw, index_type=U16),
        g.primitive(quad, [0, 1, 2, 0, 2, 3], m_metal, index_type=U8),
        g.primitive(light, [0, 1, 2], m_light, index_type=U32),
    ]
    g.node(mesh=g.mesh(prims))
    g.camera(0.9, translation=[0.0, 1.6, 2.5], rotation=[-0.0499792, 0.0, 0.0, 0.9987503])
    return g


def texall(name="texall", rough_floor=0.0):
    """`texmaps` is the same scene with every roughness at least `rough_floor` = 0.35: texall's alpha = 0.0016
    near-mirrors make the reference's own GGX D term ill-conditioned in float32 (1e-2 relative noise between any two
    operation orders), which forces a loose per-pixel bound on the path-by-path test; texmaps keeps all four texture
    maps, the alpha coverage, the node hierarchy and the index types, and is held to the tight bound."""
    rng = np.random.default_rng(7)
    g = GltfBuilder(name)
    rf = lambda r: float(max(r, rough_floor))
    size = 64
    base = checker_texture(rng, size, 8)
    alpha = np.full((size, size, 1), 255, np.uint8)
    yy, xx = np.mgrid[0:size, 0:size]
    alpha[((xx // 8 + yy // 8) % 3 == 0)] = 90
    t_base = g.texture(name + "_base.png", png_bytes(np.concatenate([base, alpha], -1)))
    # normal map: gentle waves
    nx = 0.35 * np.sin(xx * 2 * np.pi / 16.0)
    ny = 0.35 * np.cos(yy * 2 * np.pi / 12.0)
    nzc = np.sqrt(np.maximum(0.0, 1 - nx * nx - ny * ny))
    nm = np.clip((np.stack([nx, ny, nzc], -1) * 0.5 + 0.5) * 255, 0, 255).astype(np.uint8)
    t_norm = g.texture(name + "_normal.png", png_bytes(nm))
    # metallic (B) roughness (G)
    mr = np.zeros((size, size, 3), np.uint8)
    mr[..., 1] = np.clip(np.maximum(40 + 3 * xx, int(np.ceil(rough_floor * 255))), 0, 255)
    mr[..., 2] = np.where(yy < size // 2, 255, 30)
    t_mr = g.texture(name + "_mr.ppm", ppm_bytes(mr))
    em = np.zeros((size, size, 3), np.uint8)
    em[16:48, 16:48] = [255, 180, 90]
    t_em = g.texture(name + "_emissive.ppm", ppm_bytes(em))
    t_one = g.texture(name + "_1x1.ppm", ppm_bytes(np.array([[[200, 120, 60]]], np.uint8)))
    g.extensions_used.add("KHR_materials_emissive_strength")

    m_ground = g.material(pbrMetallicRoughness={"baseColorTexture": {"index": t_base},
                                                "metallicRoughnessTexture": {"index": t_mr}},
                          normalTexture={"index": t_norm})
    m_glow = g.material(pbrMetallicRoughness={"baseColorFactor": [0.2, 0.2, 0.2, 1.0], "metallicFactor": 0.0,
                                              "roughnessFactor": 0.9},
                        emissiveFactor=[1.0, 1.0, 1.0], emissiveTexture={"index": t_em},
                        extensions={"KHR_materials_emissive_strength": {"emissiveStrength": 4.0}})
    m_alpha = g.material(pbrMetallicRoughness={"baseColorFactor": [0.3, 0.6, 0.9, 0.5], "metallicFactor": 0.2,
                                               "roughnessFactor": rf(0.1)})
    m_one = g.material(pbrMetallicRoughness={"baseColorTexture": {"index": t_one}, "metallicFactor": 0.0,
                                             "roughnessFactor": rf(0.02)})
    m_mirror = g.material(pbrMetallicRoughness={"baseColorFactor": [0.9, 0.9, 0.95, 1.0], "metallicFactor": 1.0,
                                                "roughnessFactor": rf(0.0)})

    # ground: 8x8 grid, textured, with normals
    P, N, UV, T = grid(8, 8, lambda u, v: np.stack([(u - 0.5) * 8, 0.05 * np.sin(6 * u) * np.cos(5 * v), (v - 0.5) * 8], -1))
    ground = g.mesh([g.primitive(P, T[:, [0, 2, 1]], m_ground, normals=N, uv=UV * 2.5 - 0.7, index_type=U16)])
    g.node(mesh=ground)

    # glowing panel under a parent with matrix + child with TRS and non-uniform scale
    P, N, UV, T = grid(2, 2, lambda u, v: np.stack([u - 0.5, v - 0.5, np.zeros_like(u)], -1))
    panel = g.mesh([g.primitive(P, T, m_glow, normals=N, uv=UV, index_type=U8)])
    child = g.node(root=False, mesh=panel, translation=[0.0, 1.5, 0.0], rotation=[0.0, 0.3826834, 0.0, 0.9238795],
                   scale=[2.0, 1.5, 1.0])
    mat = [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, -2.0, 0.5, -1.0, 1]
    g.node(matrix=mat, children=[child])

    # alpha quad as triangle strip, no normals
    strip = np.array([[0, 0, 0], [1.5, 0, 0], [0, 1.5, 0], [1.5, 1.5, 0], [0, 3, 0.4], [1.5, 3, 0.4]], np.float32)
    g.node(mesh=g.mesh([g.primitive(strip, [0, 1, 2, 3, 4, 5], m_alpha, mode=5, index_type=U8)]),
           translation=[0.5, 0.0, 0.5])

    # 1x1-textured ball-ish blob (octahedron subdivided once) and a mirror quad
    P, N, UV, T = grid(12, 8, lambda u, v: np.stack([0.7 * np.cos(2 * np.pi * u) * np.sin(np.pi * (0.02 + 0.96 * v)),
                                                     0.7 * np.cos(np.pi * (0.02 + 0.96 * v)),
                                                     0.7 * np.sin(2 * np.pi * u) * np.sin(np.pi * (0.02 + 0.96 * v))], -1))
    g.node(mesh=g.mesh([g.primitive(P, T, m_one, normals=-N, uv=UV)]), translation=[-1.0, 0.8, 1.2],
           scale=[1.0, 1.2, 0.8])
    mq = np.array([[-3.5, 0, -3], [3.5, 0, -3], [3.5, 3, -3.4], [-3.5, 3, -3.4]], np.float32)
    g.node(mesh=g.mesh([g.primitive(mq, [0, 1, 2, 0, 2, 3], m_mirror, index_type=U32)]))

    g.camera(0.8, aspect=1.25, translation=[0.5, 2.2, 5.5], rotation=[-0.1305262, 0.0, 0.0, 0.9914449])
    return g


SCENES = {
    "tiny": tiny,
    "texall": texall,
    "texmaps": lambda: texall("texmaps", 0.35),
    "small": lambda: corridor("small", 0.1, False),
    "small_lights": lambda: corridor("small_lights", 0.1, True),
    "small_manylights": lambda: corridor("small_manylights", 0.1, True, light_res=12),  # 4 x 288 emissive triangles: a deep light BVH
    "medium_lights": lambda: corridor("medium_lights", 0.3, True),
    "big": lambda: corridor("big", 1.0, False),
    "big_lights": lambda: corridor("big_lights", 1.0, True),
}


def generate(scene, out_dir):
    return SCENES[scene]().write(out_dir)


if __name__ == "__main__":
    if len(sys.argv) != 3 or sys.argv[1] not in SCENES:
        sys.stderr.write(__doc__)
        sys.exit(2)
    print(generate(sys.argv[1], sys.argv[2]))
