#!/bin/bash
# Install the UNMODIFIED reference (a pydata/sparse checkout) into oracle/_ref/ -- git-ignored -- so that bench.py's
# reference arm times the reference's own numba path (sparse.tensordot -> _dot_csr_ndarray,
# numba_backend/_common.py:95,720-755) on the host cores, and the fuzzers in tools/ can import it.
#
#   bash oracle/make_ref.sh [<pydata/sparse checkout>]   (default: $SPARSE_REFERENCE, else /root/reference; no network)
#
# The package is pure Python (numba kernels), so the install is a copy of its `sparse/` directory.  A checkout lacks the
# setuptools-scm generated sparse/_version.py that sparse/__init__.py imports; the two-line stub below is that generated
# file, nothing else is touched.
set -euo pipefail
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
REF="${1:-${SPARSE_REFERENCE:-/root/reference}}"
DEST="$ROOT/oracle/_ref"
[ -d "$REF/sparse" ] || { echo "make_ref: $REF/sparse not found (no pydata/sparse checkout)"; exit 0; }
rm -rf "$DEST"
mkdir -p "$DEST"
cp -r "$REF/sparse" "$DEST/sparse"
chmod -R u+w "$DEST"
[ -f "$DEST/sparse/_version.py" ] || printf '__version__ = "0.0.0+ref"\n__version_tuple__ = (0, 0, 0)\n' > "$DEST/sparse/_version.py"
( cd "$DEST" && PYTHONPATH="$DEST" python -c "import sparse; print('oracle/_ref: sparse', sparse.__version__, 'backend', sparse._BACKEND)" )
