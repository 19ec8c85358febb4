#!/bin/bash
# phases of the drop-in CLI on config 4 (RT_TIMING=1)
SCENE_DIR=$(mktemp -d); trap 'rm -rf "$SCENE_DIR"' EXIT
G=$(python scenes/gen_gltf.py big_lights "$SCENE_DIR") || exit 1
for spp in 1 1000 1000; do
  s=$(date +%s%N)
  RT_TIMING=1 bin/raytracer_b200 $G 1000 1000 $spp gpurun_out/t.ppm 2>&1 | grep "raytracer_b200:\|rt_gpu:"
  e=$(date +%s%N); echo "total wall $(( (e - s) / 1000000 )) ms at $spp spp"
done
rm -f gpurun_out/t.ppm
