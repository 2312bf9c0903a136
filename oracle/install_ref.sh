#!/bin/sh
# Copy the unmodified reference package (the `audiocraft` directory of a facebookresearch/audiocraft @ 896ec7c checkout)
# into oracle/_ref (git-ignored), so that it can run on a machine that has no copy of its own, e.g. to regenerate the
# reference-CUDA golden vectors on a GPU:
#
#   sh oracle/install_ref.sh <audiocraft checkout>
#   AUDIOCRAFT_REFERENCE=oracle/_ref python tests/golden/make_golden.py fullsize_cuda
#
# Nothing is modified; oracle/ref_import.py stubs the third-party packages the import graph touches.
set -e
src=${1:-$AUDIOCRAFT_REFERENCE}
if [ -z "$src" ] || [ ! -d "$src/audiocraft/modules" ]; then
    echo "usage: $0 <path of an audiocraft checkout>" >&2
    exit 2
fi
src=$(cd "$src" && pwd)
cd "$(dirname "$0")"
rm -rf _ref
mkdir _ref
cp -R "$src/audiocraft" _ref/audiocraft
find _ref -name __pycache__ -prune -exec rm -rf {} +
