#!/bin/sh
# Build libcerb_post.so in-tree for sm_100a.  Usage: sh cerberusdet_b200/csrc/build.sh [extra nvcc flags]
#   CERB_OUT=path/to/lib.so      build a variant next to the default library (tools/ A/B runs)
#   CERB_VSRCS="decode.cu ..."   the sources the extra flags apply to (default: all of them)
# Translation units compile in parallel (make -j); objects are cached per flag set under csrc/build/.
set -e
HERE=$(cd "$(dirname "$0")" && pwd)
command -v nvcc >/dev/null 2>&1 || PATH="${CUDA_HOME:-/usr/local/cuda}/bin:$PATH"
OUT="${CERB_OUT:-$HERE/../libcerb_post.so}"
EXTRA="$*"
TAG=default
[ -z "$EXTRA" ] || TAG=$(printf '%s' "$EXTRA" | md5sum | cut -c1-10)
if [ -n "$CERB_VSRCS" ]; then
    make -s -C "$HERE" -j"$(nproc)" OUT="$OUT" TAG="$TAG" EXTRA="$EXTRA" VSRCS="$CERB_VSRCS"
else
    make -s -C "$HERE" -j"$(nproc)" OUT="$OUT" TAG="$TAG" EXTRA="$EXTRA"
fi
echo "built $OUT"
