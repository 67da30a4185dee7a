#!/usr/bin/env bash
# Test/bench infrastructure, not product: stages the UNMODIFIED reference package and its test files so that they
# travel with the working tree next to the in-tree .so files (oracle/_ref/ is git-ignored).
#
#   oracle/make_ref.sh [REFERENCE_DIR]   # copies REFERENCE_DIR/{torchsnapshot,tests} -> oracle/_ref/
#
# The reference is pure Python (setup.py:66-93 is a plain find_packages() build), so "installing" it is a copy
# of its package directory; nothing is compiled and nothing under /root/reference is written.  Used by
#   * bench.py --impl reference   (the timed reference arm: torchsnapshot.Snapshot.take/restore, snapshot.py:113,319)
#   * bench.py cpu_baseline leg   (kind "reference")
#   * tests/ -m gpu               (install() under the unmodified reference with CUDA tensors, cross-restore)
#   * tests/test_reference_suite.py (the reference's own test files run against this package, tests/ref_suite/run.py)
# Nothing under torchsnapshot_b200/ imports it.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
SRC="${1:-/root/reference}"
DST="$HERE/_ref"
if [ ! -d "$SRC/torchsnapshot" ]; then
    echo "make_ref: $SRC/torchsnapshot not found (GPU box?): keeping the existing $DST" >&2
    [ -d "$DST/torchsnapshot" ] || { echo "make_ref: no staged reference either" >&2; exit 1; }
    exit 0
fi
rm -rf "$DST"
mkdir -p "$DST"
cp -r "$SRC/torchsnapshot" "$DST/torchsnapshot"
cp -r "$SRC/tests" "$DST/tests"
find "$DST" -name '__pycache__' -type d -prune -exec rm -rf {} +
( cd "$SRC" && { git rev-parse HEAD 2>/dev/null || echo unknown; } ) > "$DST/REF_COMMIT"
# sha256 of every file of the SOURCE package, so that a run can prove the staged copy is the unmodified tree
( cd "$SRC/torchsnapshot" && find . -name '__pycache__' -prune -o -type f -print | sort | xargs sha256sum ) > "$DST/MANIFEST.sha256"
echo "make_ref: staged $(find "$DST/torchsnapshot" -name '*.py' | wc -l) python files and $(find "$DST/tests" -name 'test_*.py' | wc -l) test files from $SRC into $DST"
