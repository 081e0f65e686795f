#!/bin/bash
# ORACLE -- TEST INFRASTRUCTURE ONLY.
# Builds the REFERENCE's own closest-point extension (thirdparty/mesh_grid/{mesh_grid.cpp,
# mesh_grid_kernel.cu,matrix.h}) for sm_100a from the sources where they lie in the reference checkout
# (BODYFIT_REFERENCE, else a directory `reference` beside this repository), into oracle/_ref/
# (git-ignored, like our own .so); without a checkout it does nothing.  Nothing is copied
# into the repository: the sources are staged in a temporary directory, where the one mechanical
# patch torch >= 2 needs is applied (X.type() -> X.scalar_type() inside AT_DISPATCH_FLOATING_TYPES).
# Used only by tests as a second referee for bf_grid_nearest (distances, not face ids).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
REF="${BODYFIT_REFERENCE:-$HERE/../../reference}/thirdparty/mesh_grid"
OUT="$HERE/_ref"
[ -d "$REF" ] || { echo "no reference checkout ($REF), skipping"; exit 0; }
if [ -n "$(ls "$OUT"/mesh_grid*.so 2>/dev/null)" ] && [ "$1" != "-f" ]; then echo "oracle/_ref already built"; exit 0; fi
TMP="$(mktemp -d /tmp/bf_ref_build.XXXXXX)"
cp "$REF/mesh_grid.cpp" "$REF/mesh_grid_kernel.cu" "$REF/matrix.h" "$REF/setup.py" "$TMP/"
sed -i -E 's/AT_DISPATCH_FLOATING_TYPES\((verts|image|faces)\.type\(\)/AT_DISPATCH_FLOATING_TYPES(\1.scalar_type()/' "$TMP/mesh_grid_kernel.cu"
(cd "$TMP" && TORCH_CUDA_ARCH_LIST="10.0a" MAX_JOBS=4 python setup.py build_ext --inplace > build.log 2>&1) || { tail -30 "$TMP/build.log"; exit 1; }
mkdir -p "$OUT"
cp "$TMP"/mesh_grid*.so "$OUT/"
rm -rf "$TMP"
ls -la "$OUT"
