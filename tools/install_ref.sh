#!/usr/bin/env bash
# Install the UNMODIFIED reference (chzhang18/RAG, pure Python, no setup.py -> nothing to pip-install)
# at oracle/_ref/, inside the tree, so that it goes wherever the built tree goes (like the built .so files).
#   oracle/_ref/ is git-ignored (the reference's sources never enter this repo's history).
#   Only src/ is needed: models/, automl/, approaches/, utils.py, utilstool/.
# Run by __graft_entry__.build(); exits 3 and leaves oracle/_ref/ as it is when there is no checkout to install.
# Used by: tests/test_reference_network_gpu.py (drop-in proven on the real Network / BasicNetwork),
#          smoke(), bench.py --impl reference and bench.py's cpu_baseline / torch_cuda_reference legs.
set -euo pipefail
ROOT="$(cd "$(dirname "${BASH_SOURCE[0]}")/.." && pwd)"
SRC="${RAG_REFERENCE:-/root/reference}"
DST="$ROOT/oracle/_ref"
if [ ! -d "$SRC/src/models" ]; then
  echo "install_ref: $SRC/src not found (set RAG_REFERENCE to a checkout of the reference)" >&2
  exit 3
fi
rm -rf "$DST"
mkdir -p "$DST"
cp -r "$SRC/src" "$DST/src"
find "$DST" -name '__pycache__' -type d -prune -exec rm -rf {} +
# record what was installed: file list + sha256, so a test can prove the copy is unmodified
( cd "$DST/src" && find . -type f -name '*.py' | sort | xargs sha256sum ) > "$DST/MANIFEST.sha256"
echo "installed $(wc -l < "$DST/MANIFEST.sha256") reference files into $DST"
