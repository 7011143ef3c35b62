#!/bin/bash
# build_ref_runtime.sh -- builds the REFERENCE runtime (ICLDisco/parsec, unmodified sources from /root/reference) plus
# this repository's MCA device component into oracle/_ref/parsec (git-ignored; travels to the GPU box).
#
#   * the reference tree is copied to a scratch overlay (it is read-only where it lies) and the ONLY thing added is the
#     directory parsec/mca/device/b200/ (our component; static MCA components have to live in the tree, SURVEY.md 8b);
#   * hwloc: the image has none and the runtime does not link without one at this commit (SURVEY.md 8c); the
#     flat-topology shim of oracle/hwloc_shim/ stands in (test infrastructure);
#   * PARSEC_GPU_WITH_CUDA=ON so that parsec-ptgpp emits BODY [type=CUDA] hooks (PARSEC_HAVE_DEV_CUDA_SUPPORT) and the
#     reference's own CUDA component is available as a second baseline on the GPU box.
# Outputs: oracle/_ref/parsec/{lib/libparsec.so*,bin/parsec-ptgpp,include/...}.  Needs cmake + ninja (both in the image).
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
REF=${REF:-/root/reference}
# one scratch tree per user and checkout: its CMake cache holds this checkout's paths (PB2_ROOT, the install prefix)
SCRATCH=${SCRATCH:-${TMPDIR:-/tmp}/pb2_ref-$(id -u)-$(printf %s "$ROOT" | md5sum | cut -c1-12)}
PREFIX=$ROOT/oracle/_ref/parsec
[ -d "$REF/parsec" ] || { echo "no reference tree at $REF: keeping the prebuilt oracle/_ref"; exit 0; }
[ -f "$ROOT/parsec_b200/libparsec_b200.so" ] || { echo "build parsec_b200/libparsec_b200.so first (make)"; exit 1; }
mkdir -p "$SCRATCH/hwloc/include" "$SCRATCH/hwloc/lib"
if [ ! -d "$SCRATCH/src/parsec" ]; then cp -r "$REF" "$SCRATCH/src"; chmod -R u+w "$SCRATCH/src"; fi
rm -rf "$SCRATCH/src/parsec/mca/device/b200"
mkdir -p "$SCRATCH/src/parsec/mca/device/b200"
cp "$ROOT"/parsec_b200/mca/b200/* "$SCRATCH/src/parsec/mca/device/b200/"
gcc -O2 -fPIC -c -o "$SCRATCH/hwloc/hwloc_shim.o" "$ROOT/oracle/hwloc_shim/hwloc_shim.c"
ar rcs "$SCRATCH/hwloc/lib/libhwloc.a" "$SCRATCH/hwloc/hwloc_shim.o"
cp "$ROOT/oracle/hwloc_shim/hwloc.h" "$SCRATCH/hwloc/include/"
if [ ! -f "$SCRATCH/build/build.ninja" ] || [ "$1" = "--reconfigure" ]; then
  cmake -G Ninja -S "$SCRATCH/src" -B "$SCRATCH/build" -DCMAKE_BUILD_TYPE=Release -DBUILD_TESTING=OFF \
    -DPARSEC_DIST_WITH_MPI=OFF -DPARSEC_GPU_WITH_CUDA=ON -DPARSEC_GPU_WITH_HIP=OFF -DPARSEC_GPU_WITH_LEVEL_ZERO=OFF \
    -DPARSEC_WITH_DEVEL_HEADERS=ON -DBUILD_SHARED_LIBS=ON \
    -DCMAKE_CUDA_COMPILER=/usr/local/cuda/bin/nvcc -DCUDAToolkit_ROOT=/usr/local/cuda \
    -DHWLOC_ROOT="$SCRATCH/hwloc" -DCMAKE_PREFIX_PATH="$SCRATCH/hwloc" \
    -DPB2_ROOT="$ROOT" -DCMAKE_INSTALL_PREFIX="$PREFIX" \
    -DCMAKE_PROJECT_PARSEC_INCLUDE="$ROOT/oracle/ref_rpath.cmake" > "$SCRATCH/configure.log" 2>&1 \
    || { tail -30 "$SCRATCH/configure.log"; exit 1; }
  grep -E "Module .b200|Active modules for the device" "$SCRATCH/configure.log" || true
fi
ninja -C "$SCRATCH/build" > "$SCRATCH/build.log" 2>&1 || { grep -E "error|Error" -A3 "$SCRATCH/build.log" | head -60; exit 1; }
rm -rf "$PREFIX"
cmake --install "$SCRATCH/build" > "$SCRATCH/install.log" 2>&1 || { tail -20 "$SCRATCH/install.log"; exit 1; }
# the shim's header is needed by whoever includes parsec's devel headers
cp "$ROOT/oracle/hwloc_shim/hwloc.h" "$PREFIX/include/"
# the install travels to other machines by copies that may drop symbolic links (libparsec.so.4 -> libparsec.so.4.1.0,
# the name the applications load): turn every link into a copy of its target
find "$PREFIX" -type l | while read -r l; do t=$(readlink -f "$l"); rm "$l"; cp "$t" "$l"; done
# and for the same reason the RUNPATH of libparsec (ref_rpath.cmake) must not name this checkout
if readelf -d "$PREFIX/lib/libparsec.so" | grep -F "$ROOT"; then echo "libparsec.so has an absolute RUNPATH: run $0 --reconfigure"; exit 1; fi
du -sh "$PREFIX" | sed 's/^/installed: /'
