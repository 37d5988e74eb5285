#!/bin/bash
# Recipe for oracle/_ref: the UNMODIFIED reference (torchkge, pure Python) installed from its own
# sources where they lie under /root/reference, outputs only into oracle/_ref/ (git-ignored, shipped
# to the GPU box with the snapshot).  Used as the checker / CPU baseline only (bench.py
# cpu_baseline.kind = "reference", --impl reference); nothing in torchkge_b200 imports it.
# /root/reference is read-only and setuptools writes an egg-info next to setup.py, so the install runs
# from a scratch copy; no dependency is fetched (--no-index --no-deps: torch, pandas, tqdm are in the image).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
REF="${1:-/root/reference}"
[ -d "$REF/torchkge" ] || { echo "make_ref: $REF/torchkge not found (nothing to do)"; exit 0; }
TMP="$(mktemp -d)"
trap 'rm -rf "$TMP"' EXIT
# copies keep the sources' read-only modes: make them writable, so that they can be replaced and removed
cp -r "$REF" "$TMP/src" && chmod -R u+w "$TMP/src"
if [ -d "$HERE/_ref" ]; then chmod -R u+w "$HERE/_ref"; fi
rm -rf "$HERE/_ref"
python -m pip install --quiet --no-index --no-build-isolation --no-deps --no-compile \
    --target "$HERE/_ref" "$TMP/src" 2>"$TMP/pip.log" || {
  # a plain copy of the package directory is the same thing for a pure-Python package
  echo "make_ref: pip install failed ($(tail -1 "$TMP/pip.log")); copying the package directory"
  mkdir -p "$HERE/_ref" && cp -r "$REF/torchkge" "$HERE/_ref/torchkge" && chmod -R u+w "$HERE/_ref"
}
python - <<PY
import sys
sys.path.insert(0, "$HERE/_ref")
import torchkge
print("oracle/_ref: torchkge", torchkge.__version__, "from", torchkge.__file__)
PY
