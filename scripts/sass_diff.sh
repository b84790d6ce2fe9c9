#!/usr/bin/env bash
# SASS of every kernel of the working tree against a git revision (default: HEAD~1), object by object.  Both sides are compiled
# with slam3d_b200/build.py's flags in temporary directories; the source path in cuobjdump's `identifier` line and the
# anonymous-namespace hash nvcc derives from it are masked, everything else must match.  No GPU needed.
#     scripts/sass_diff.sh [revision]
set -euo pipefail
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
REV="${1:-HEAD~1}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
CUOBJDUMP="$(dirname "$NVCC")/cuobjdump"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC,-O2)
TMP="$(mktemp -d)"
trap 'rm -rf "$TMP"' EXIT
mkdir -p "$TMP/old" "$TMP/new"
git -C "$ROOT" archive "$REV" slam3d_b200/csrc include | tar -x -C "$TMP/old"
cp -r "$ROOT/slam3d_b200" "$ROOT/include" "$TMP/new/"
status=0
for f in voxel grid knn gicp ndt map ransac api; do
  for side in old new; do
    (cd "$TMP/$side/slam3d_b200/csrc" && "$NVCC" "${FLAGS[@]}" -c "$f.cu" -o "$TMP/$side/$f.o")
    "$CUOBJDUMP" -sass "$TMP/$side/$f.o" | grep -v '^[[:space:]]*identifier' | sed 's/_GLOBAL__N__[0-9a-f]*_/_GLOBAL__N__/g' > "$TMP/$side/$f.sass"
  done
  kernels=$(grep -c 'Function :' "$TMP/old/$f.sass" || true)
  if cmp -s "$TMP/old/$f.sass" "$TMP/new/$f.sass"; then echo "$f.cu: SASS identical ($kernels kernels)"
  else echo "$f.cu: SASS differs"; diff "$TMP/old/$f.sass" "$TMP/new/$f.sass" | head -20; status=1; fi
done
exit $status
