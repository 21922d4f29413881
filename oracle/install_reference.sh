#!/bin/bash
# Install the UNMODIFIED reference (brandondube/prysm v0.22, pure Python) into oracle/_ref/ (git-ignored).
#   bash oracle/install_reference.sh <prysm source tree>
# It serves `bench.py --impl reference`, bench.py's cpu_baseline and the drop-in tests that patch the real prysm.
# The reference's build backend (hatchling) may not be installed and an offline machine cannot fetch it.  The package
# is pure Python and its wheel target is `packages = ["prysm"]`, so the same files are installed by building from a
# scratch copy whose [build-system] stanza names setuptools instead; not one line of the prysm/ package is touched
# (checked below with diff -r).
set -euo pipefail
HERE="$(cd "$(dirname "$0")" && pwd)"
SRC="${1:?usage: install_reference.sh <prysm source tree>}"
DST="$HERE/_ref"
TMP="$(mktemp -d)"
trap 'rm -rf "$TMP"' EXIT
cp -r "$SRC/prysm" "$TMP/prysm"
cp "$SRC/LICENSE.md" "$SRC/README.md" "$TMP/" 2>/dev/null || true
cat > "$TMP/pyproject.toml" <<'TOML'
[build-system]
requires = ["setuptools"]
build-backend = "setuptools.build_meta"
[project]
name = "prysm"
version = "0.22"
dependencies = []
[tool.setuptools.packages.find]
include = ["prysm*"]
[tool.setuptools.package-data]
"*" = ["*"]
TOML
rm -rf "$DST"
python -m pip install --no-index --no-build-isolation --no-deps --target "$DST" "$TMP" 2>&1 | tail -2
diff -r -q "$SRC/prysm" "$DST/prysm" -x __pycache__ && echo "oracle/_ref/prysm is identical to $SRC/prysm"
