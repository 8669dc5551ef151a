#!/bin/bash
# Recipe for oracle/_ref/: the reference's own hot-path files, copied VERBATIM from the read-only reference checkout into the
# git-ignored oracle/_ref/ (never committed; it travels to the GPU box with the gpurun snapshot like a built .so).  bench.py's
# `--impl reference` arm and the dss2_run.py exec test run these files over oracle/pyg_shim (torch_geometric is not installable
# here).  Nothing in the product package reads oracle/_ref/.
#   usage: tools/make_oracle_ref.sh [reference_root]        (default: $DSS2_REFERENCE)
set -e
REF="${1:-${DSS2_REFERENCE:-}}"
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
DST="$ROOT/oracle/_ref"
if [ -z "$REF" ] || [ ! -f "$REF/networks.py" ]; then
  echo "make_oracle_ref: no reference checkout (argument or DSS2_REFERENCE: '$REF'); keeping whatever is in $DST" >&2
  exit 0
fi
mkdir -p "$DST"
for f in networks.py data.py dss2_run.py loadsampling.py; do
  cp -f "$REF/$f" "$DST/$f" && chmod 644 "$DST/$f"
done
( cd "$REF" && sha256sum networks.py data.py dss2_run.py loadsampling.py ) > "$DST/SHA256SUMS"
echo "make_oracle_ref: copied networks.py data.py dss2_run.py loadsampling.py -> $DST"
