#!/bin/bash
# Install the UNMODIFIED reference (jeanfeydy/geomloss @ 00e493f, pure Python) into oracle/_ref/ so that it travels to
# the GPU box with the repository snapshot (oracle/_ref/ is git-ignored, not gpurun-ignored):
#
#     bash oracle/make_ref.sh            # needs /root/reference (build container only)
#
# Nothing is copied into the tracked tree: pip builds a wheel from a scratch copy under /tmp (the reference mount is
# read-only) and unpacks it under oracle/_ref/.  Used by
#   * bench.py --impl reference  ->  cpu_baseline.kind = "reference": the reference's own softmin_tensorized /
#     cost routines timed on the host cores.
set -euo pipefail
HERE="$(cd "$(dirname "$0")" && pwd)"
SRC="${GEOMLOSS_REFERENCE_ROOT:-/root/reference}"
if [ ! -d "$SRC/src/geomloss" ]; then
  echo "make_ref: $SRC not found (GPU box?): keeping whatever is in $HERE/_ref" >&2
  exit 0
fi
TMP="$(mktemp -d /tmp/geomloss_ref.XXXXXX)"
trap 'rm -rf "$TMP"' EXIT
cp -r "$SRC" "$TMP/reference"
rm -rf "$HERE/_ref"
mkdir -p "$HERE/_ref"
python -m pip install --quiet --no-index --no-build-isolation --no-deps --find-links /opt/wheelhouse \
  --target "$HERE/_ref" "$TMP/reference" 2> "$TMP/pip.log" || { cat "$TMP/pip.log" >&2; exit 1; }
python - <<PY
import sys
sys.path.insert(0, "$HERE/_ref")
import geomloss
print("oracle/_ref: geomloss", geomloss.__version__, "from", geomloss.__file__)
PY
