#!/usr/bin/env bash
# Build the UNMODIFIED reference (pymc-devs/pytensor) into oracle/_ref so that it can
#  (a) host the CUDALinker plugin (PyTensor is the host: graph IR, rewrites, pytensor.function), and
#  (b) act as the parity oracle / CPU baseline through its own C linker (mode='CVM').
#
# `pip install --target oracle/_ref <pytensor checkout>` needs `versioneer` (setup.py imports it), which may not be
# installable offline.  This recipe does what that install would do: copy the package tree and build the one compiled
# extension (pytensor/scan/scan_perform.pyx, setup.py:24-29) with cython + gcc.  Nothing is written into the checkout;
# the output directory is git-ignored (it is NOT product source).
#   usage: bash oracle/build_ref.sh [pytensor checkout, default /root/reference]
set -euo pipefail
REF=${1:-/root/reference}
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")/.." && pwd)"
OUT="$HERE/oracle/_ref"
if [ ! -d "$REF/pytensor" ]; then
  echo "pytensor checkout not found at $REF: nothing to build"; exit 0
fi
rm -rf "$OUT"; mkdir -p "$OUT"
# the checkout may be read-only: the copy must not inherit its modes, or the extension cannot be written into it
cp -r --no-preserve=mode,ownership "$REF/pytensor" "$OUT/pytensor"
find "$OUT" -name '__pycache__' -type d -prune -exec rm -rf {} +
PYINC=$(python -c "import sysconfig; print(sysconfig.get_paths()['include'])")
NPINC=$(python -c "import numpy; print(numpy.get_include())")
EXT=$(python -c "import sysconfig; print(sysconfig.get_config_var('EXT_SUFFIX'))")
TMP=$(mktemp -d)
cp "$REF/pytensor/scan/scan_perform.pyx" "$TMP/"
chmod u+w "$TMP/scan_perform.pyx"
( cd "$TMP" && cython -3 scan_perform.pyx -o scan_perform.c )
gcc -O2 -shared -fPIC -fno-strict-aliasing -DNPY_NO_DEPRECATED_API=NPY_1_7_API_VERSION \
    -I"$PYINC" -I"$NPINC" "$TMP/scan_perform.c" -o "$OUT/pytensor/scan/scan_perform$EXT"
rm -rf "$TMP"
echo "reference built into $OUT"
