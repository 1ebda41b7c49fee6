#!/usr/bin/env bash
# build_ref.sh — TEST INFRASTRUCTURE.  Compiles the UNMODIFIED reference core from
# a checkout of it (read-only; not part of this repository): the one
# MCSKIN_REFERENCE_DIR names, else `reference` beside this repository.  Adds
# oracle/ref_shim.cpp and links oracle/_ref/libmcskin_ref.so.  Only outputs land
# under oracle/_ref/ (git-ignored).
#
# Flags = the reference's Release configuration (scripts/package.sh:57 ->
# CMAKE_BUILD_TYPE=Release -> -O3 -DNDEBUG, C++17, no -march, no fast-math), i.e.
# x86-64 baseline: no FMA contraction, IEEE div/sqrt, glibc libm, libstdc++ <random>.
# The reference's own CMake build is not run (it needs Qt6 and FetchContent).
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="$HERE/_ref"
if [ -n "${MCSKIN_REFERENCE_DIR:-}" ]; then
    REF="$MCSKIN_REFERENCE_DIR"
    if [ ! -d "$REF/src" ]; then
        echo "build_ref.sh: MCSKIN_REFERENCE_DIR=$REF is not a checkout of the reference (no src/)" >&2
        exit 1
    fi
else
    # default: a checkout named `reference` beside this repository; absent or unreadable means not present
    REF="$HERE/../../reference"
    if [ ! -d "$REF/src" ] || [ ! -r "$REF/src" ]; then
        echo "build_ref.sh: no checkout of the reference at $REF (set MCSKIN_REFERENCE_DIR); keeping any prebuilt $OUT" >&2
        exit 0
    fi
fi
mkdir -p "$OUT/obj"
CXX="${CXX:-g++}"
CXXFLAGS="-std=c++17 -O3 -DNDEBUG -fPIC -fno-fast-math -ffp-contract=off -I$REF/src -I$REF/third_party"
# src/CMakeLists.txt:2-14 CORE_SOURCES, minus gui/camera_controller.cpp (UI state, not on the path)
SOURCES="skin/stb_impl.cpp skin/image.cpp skin/skin_parser.cpp scene/mesh_builder.cpp scene/camera.cpp
raytracer/intersection.cpp raytracer/shading.cpp raytracer/raytracer.cpp raytracer/tile_renderer.cpp
output/image_writer.cpp"
OBJS=""
for s in $SOURCES; do
    o="$OUT/obj/$(echo "$s" | tr '/' '_' | sed 's/\.cpp$/.o/')"
    if [ ! -f "$o" ] || [ "$REF/src/$s" -nt "$o" ]; then
        $CXX $CXXFLAGS -c "$REF/src/$s" -o "$o" &
    fi
    OBJS="$OBJS $o"
done
wait
$CXX $CXXFLAGS -I"$HERE/../include" -c "$HERE/ref_shim.cpp" -o "$OUT/obj/ref_shim.o"
# --wrap counts intersectScene invocations (the "ray" unit of BASELINE.md) without touching the sources
$CXX -shared -o "$OUT/libmcskin_ref.so" $OBJS "$OUT/obj/ref_shim.o" \
    -Wl,--wrap=_Z14intersectSceneRK3RayRK5Scene -lpthread
echo "built $OUT/libmcskin_ref.so"
