#!/bin/bash
# CLI wall times on the GPU box: the drop-in (bin/raytracer_b200) on BASELINE config 4, with and without the reference's
# scene-BVH build, and the unmodified reference binary (oracle/_ref/raytracer) at 1 and 5 spp (its 1000 spp would take ~5 min
# on 16 cores; load + BVH build is the intercept, the slope is per spp).
mkdir -p gpurun_out
OUT=gpurun_out/r2_cli_times.log
: > $OUT
SCENE_DIR=$(mktemp -d); trap 'rm -rf "$SCENE_DIR"' EXIT
G=$(python scenes/gen_gltf.py big_lights "$SCENE_DIR") || exit 1
t() { local s=$(date +%s%N); "$@" > /dev/null 2> gpurun_out/cli.err; local rc=$?; local e=$(date +%s%N); echo "$(( (e - s) / 1000000 )) ms  rc=$rc  : ${ENVDESC} $*" | tee -a $OUT; tail -1 gpurun_out/cli.err >> $OUT; }
nproc | sed 's/^/host cores: /' | tee -a $OUT
ENVDESC="" t bin/raytracer_b200 $G 1000 1000 1000 gpurun_out/cli_c4.ppm
ENVDESC="" t bin/raytracer_b200 $G 1000 1000 1000 gpurun_out/cli_c4.ppm
export RT_HOST_SCENE_BVH=1; ENVDESC="RT_HOST_SCENE_BVH=1" t bin/raytracer_b200 $G 1000 1000 1000 gpurun_out/cli_c4_hostbvh.ppm; unset RT_HOST_SCENE_BVH
ENVDESC="" t bin/raytracer_b200 $G 1000 1000 1 gpurun_out/cli_1spp.ppm
ENVDESC="" t python -m rt_b200.cli $G 1000 1000 1000 gpurun_out/cli_py.ppm
ENVDESC="(reference)" t oracle/_ref/raytracer $G 1000 1000 1 gpurun_out/ref_1spp.ppm
ENVDESC="(reference)" t oracle/_ref/raytracer $G 1000 1000 5 gpurun_out/ref_5spp.ppm
cmp gpurun_out/cli_c4.ppm gpurun_out/cli_c4_hostbvh.ppm && echo "drop-in PPM identical with and without the host scene BVH" | tee -a $OUT
rm -f gpurun_out/*.ppm
cat $OUT
