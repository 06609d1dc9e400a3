#!/bin/sh
# tests/golden/sleeping.rtsc.gz: RayTracing/Data/sleeping (372 triangles, one 512x512 RGB texture, DIFFUSE / SPECULAR /
# LIGHT / TEXTURE materials) as decoded by the REFERENCE's own loader — getTrianglesData_ (mesh.h:279-613) and stb_image,
# compiled from where they lie into oracle/_ref/ref_host — written in the host library's RTSC container and gzipped.
# An output of the reference (REF, default $RT_REFERENCE: a reference checkout), committed so that the
# loader -> GPU parity test runs on the GPU box, which has no reference tree.
set -e
HERE=$(cd "$(dirname "$0")/../.." && pwd)
REF=${REF:-$RT_REFERENCE}
"$HERE/oracle/_ref/ref_host" load "$REF/RayTracing/Data/sleeping" none /tmp/sleeping.rtsc
gzip -9 -n -c /tmp/sleeping.rtsc > "$HERE/tests/golden/sleeping.rtsc.gz"
ls -la "$HERE/tests/golden/sleeping.rtsc.gz"
