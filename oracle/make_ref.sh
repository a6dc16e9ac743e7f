#!/bin/bash
# Install the UNMODIFIED reference into oracle/_ref so that `bench.py --impl reference` and the bench's cpu_baseline
# legs time the reference's own code on the host cores (cpu_baseline.kind = "reference").  oracle/_ref is git-ignored:
# no reference sources enter this repository's history.  MONAI itself is not installable offline: the reference's
# imports of it resolve to oracle/monai_shim (thin Convolution / MLPBlock / transform wrappers restated from SURVEY.md
# section 8c).  Does nothing where the reference source tree (REFERENCE_DIR) is absent.
set -euo pipefail
here="$(cd "$(dirname "$0")" && pwd)"
ref=${REFERENCE_DIR:-/root/reference}
dst="$here/_ref"
[ -f "$ref/setup.py" ] || { echo "make_ref: $ref not present"; exit 0; }
tmp=$(mktemp -d)
cp -r "$ref" "$tmp/src"                      # the build writes egg-info into the source tree, which may be read-only
chmod -R u+w "$tmp/src"                      # cp keeps the source's modes
rm -rf "$dst"
mkdir -p "$dst"
python -m pip install --quiet --no-index --no-build-isolation --no-deps --target "$dst" "$tmp/src"
rm -rf "$dst/tests" "$tmp"                   # the reference's own `tests` package would shadow this repository's
echo "installed $(ls "$dst" | tr '\n' ' ')into oracle/_ref"
