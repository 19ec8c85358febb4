"""Digest of a flattened scene (rt_b200.SceneData): pins a scene too large to store as golden data
(tests/golden/big_lights_flat.json, written by tests/golden/make_golden.py, checked by tests/test_host.py)."""
import hashlib

import numpy as np

SECTIONS = ["tri_pos", "tri_normals", "tri_uv", "tri_tangents", "tri_material", "materials", "textures", "texels",
            "scene nodes", "scene objects", "light nodes", "light objects"]
FIELDS = ["camera_position", "camera_right", "camera_up", "camera_forward", "fov_x", "bg_color", "eps", "min_roughness",
          "vndf_factor"]


def flattening_digest(sc):
    """sha256 of every section of a flattened scene, with its scalar fields."""
    fields = {k: np.asarray(getattr(sc, k)).tolist() for k in FIELDS}
    fields.update(ray_depth=int(sc.ray_depth), env_texture=int(sc.env_texture), scene_root=int(sc.scene_bvh.root),
                  light_root=int(sc.light_bvh.root))
    sections = {name: None if x is None else hashlib.sha256(x.tobytes()).hexdigest() for x, name in zip(sc._sections(), SECTIONS)}
    return {"n_tris": int(sc.n_tris), "sections": sections, "fields": fields}
