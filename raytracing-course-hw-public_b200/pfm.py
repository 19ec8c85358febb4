"""Portable float maps (PFM): "PF" for 3 channels, "Pf" for 1, little-endian (scale -1), rows bottom to top.  The
AOV buffers of the CLIs (RT_AOV) are written in this format."""
import os

import numpy as np


def write_pfm(path, img):
    """float32 [H, W, 3] or [H, W] -> path"""
    img = np.asarray(img, np.float32)
    if img.ndim == 3 and img.shape[2] == 3:
        tag = b"PF"
    elif img.ndim == 2:
        tag = b"Pf"
    else:
        raise ValueError(f"write_pfm: expected [H, W, 3] or [H, W], got {img.shape}")
    h, w = img.shape[:2]
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "wb") as f:
        f.write(tag + b"\n%d %d\n-1\n" % (w, h))
        f.write(np.ascontiguousarray(img[::-1], "<f4").tobytes())


def read_pfm(path):
    """path -> float32 [H, W, 3] ("PF") or [H, W] ("Pf"), top row first"""
    with open(path, "rb") as f:
        data = f.read()
    lines, off = [], 0
    while len(lines) < 3:  # tag, "width height", scale: three whitespace-terminated lines
        end = data.index(b"\n", off)
        lines.append(data[off:end].strip())
        off = end + 1
    tag, (w, h), scale = lines[0], map(int, lines[1].split()), float(lines[2])
    if tag not in (b"PF", b"Pf"):
        raise ValueError(f"{path}: not a PFM file")
    c = 3 if tag == b"PF" else 1
    img = np.frombuffer(data, "<f4" if scale < 0 else ">f4", count=w * h * c, offset=off).astype(np.float32)
    img = img.reshape((h, w, 3) if c == 3 else (h, w))
    return np.ascontiguousarray(img[::-1])
