"""glTF files for the multi-view tests, written from a gen_gltf scene: the same geometry with two more camera nodes
traversed before the scene's own camera, so that camera stays the last one (the one the loader keeps)."""
import json
import os

import numpy as np


def yawed(cam, degrees):
    """`cam` turned about its own up axis by `degrees` (float32)."""
    import rt_b200

    t = np.radians(degrees)
    c, s = np.float32(np.cos(t)), np.float32(np.sin(t))
    return rt_b200.Camera(cam.position, c * cam.right - s * cam.forward, cam.up, c * cam.forward + s * cam.right, cam.fov_x)


def with_three_cameras(src, out_name):
    """Three camera nodes in traversal order: (0) the scene's camera under a parent node moved 0.4 along x, (1) a
    narrower camera 0.3 higher, (2) the scene's own camera.  Returns the path of the new file (next to `src`, whose
    buffers and images it shares)."""
    with open(src) as f:
        doc = json.load(f)
    nodes = doc["nodes"]
    own = next(n for n in nodes if "camera" in n)
    persp = doc["cameras"][own["camera"]]["perspective"]
    doc["cameras"].append({"type": "perspective", "perspective": dict(persp, yfov=persp["yfov"] * 0.7)})
    moved = dict(own)
    nodes.append(moved)
    nodes.append({"translation": [0.4, 0.0, 0.0], "children": [len(nodes) - 1]})
    higher = dict(own, camera=len(doc["cameras"]) - 1)
    t = own.get("translation", [0.0, 0.0, 0.0])
    higher["translation"] = [t[0], t[1] + 0.3, t[2]]
    nodes.append(higher)
    doc["scenes"][doc.get("scene", 0)]["nodes"] = [len(nodes) - 2, len(nodes) - 1] + doc["scenes"][doc.get("scene", 0)]["nodes"]
    out = os.path.join(os.path.dirname(src), out_name)
    with open(out, "w") as f:
        json.dump(doc, f)
    return out


def without_cameras(src, out_name):
    """The same scene without any camera node."""
    with open(src) as f:
        doc = json.load(f)
    scene = doc["scenes"][doc.get("scene", 0)]
    scene["nodes"] = [i for i in scene["nodes"] if "camera" not in doc["nodes"][i]]
    out = os.path.join(os.path.dirname(src), out_name)
    with open(out, "w") as f:
        json.dump(doc, f)
    return out
