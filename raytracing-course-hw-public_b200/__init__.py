"""B200-native path-tracing backend for firelion9/raytracing-course-hw-public (hot path only).

Python mirror of the host side: scene flattening (`SceneData`), the ctypes binding of the CUDA C ABI
(`gpu.RtGpu`, include/rt_gpu.h) and host helpers (`host`).  The compute lives in csrc/ (CUDA, sm_100a).
"""
from ._abi import (RT_FLAG_ACCUMULATE, RT_MODE_BEAUTY, RT_MODE_PRIMARY_IDS, RT_NO_CHILD, BvhData, Camera, Projection, SceneData)

__all__ = ["SceneData", "BvhData", "Camera", "Projection", "RT_NO_CHILD", "RT_MODE_BEAUTY", "RT_MODE_PRIMARY_IDS", "RT_FLAG_ACCUMULATE"]
