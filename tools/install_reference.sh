#!/usr/bin/env bash
# Install the UNMODIFIED reference (yakvrz/minesweeper-ppo) into baseline/_ref/.
#
#   tools/install_reference.sh <checkout of the reference>     (or MSW_REFERENCE_SRC=<checkout>)
#
# The reference has no setup.py / pyproject.toml (its scripts run with PYTHONPATH=., README.md:28-32),
# so "install" = a verbatim copy of the tree.  baseline/_ref/ is git-ignored (never part of this
# repo's history).  With it present
#   * tests/test_gpu_reference_live.py drives it lock-step against the CUDA env,
#   * the reference-comparison tests that otherwise skip run, and
#   * bench.py times its numba env on the host cores (cpu_baseline.reference_numba).
set -euo pipefail
SRC="${1:-${MSW_REFERENCE_SRC:-}}"
ROOT="$(cd "$(dirname "${BASH_SOURCE[0]}")/.." && pwd)"
DST="$ROOT/baseline/_ref"
if [ -z "$SRC" ] || [ ! -d "$SRC/minesweeper" ]; then
  echo "install_reference: '$SRC' is not a checkout of the reference (usage: $0 <checkout>)" >&2
  exit 3
fi
rm -rf "$DST.tmp"
mkdir -p "$DST.tmp"
# sources only: no caches, no web UI assets, no docs
( cd "$SRC" && find . -type f \( -name '*.py' -o -name '*.yaml' -o -name 'requirements.txt' \) \
    -not -path './webui/*' -not -path '*/__pycache__/*' -print0 | cpio -0 -pdm --quiet "$DST.tmp" ) 2>/dev/null \
  || ( cd "$SRC" && find . -type f \( -name '*.py' -o -name '*.yaml' -o -name 'requirements.txt' \) \
    -not -path './webui/*' -not -path '*/__pycache__/*' | while read -r f; do mkdir -p "$DST.tmp/$(dirname "$f")"; cp "$f" "$DST.tmp/$f"; done )
( cd "$SRC" && find . -type f -name '*.py' -not -path './webui/*' -not -path '*/__pycache__/*' | sort | xargs sha256sum ) > "$DST.tmp/SHA256SUMS"
rm -rf "$DST"
mv "$DST.tmp" "$DST"
echo "installed reference into $DST ($(find "$DST" -name '*.py' | wc -l) python files)"
