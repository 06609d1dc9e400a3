#!/bin/sh
# Real-asset scenes for BASELINE config 2(i): the reference's own loader + stb (through the harness
# oracle/_ref/ref_host, built from the reference checkout REF, default $RT_REFERENCE) decode RayTracing/Data/<model> into an RTSC file the
# host library can read (rth_scene_load).  Output is git-ignored (60 MB for `robot`: a 4096^2 texture).
set -e
HERE=$(cd "$(dirname "$0")/.." && pwd)
REF=${REF:-$RT_REFERENCE}
mkdir -p "$HERE/assets/_gen"
for m in ${@:-robot}; do
  "$HERE/oracle/_ref/ref_host" load "$REF/RayTracing/Data/$m" none "$HERE/assets/_gen/$m.rtsc"
  ls -la "$HERE/assets/_gen/$m.rtsc"
done
