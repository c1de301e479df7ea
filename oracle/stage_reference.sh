#!/bin/bash
# Stages the UNMODIFIED reference (ekzhu/datasketch) from a checkout of it into the git-ignored oracle/_ref/:
#   oracle/_ref/site/      the reference package, installed for `bench.py --impl reference` and bench.py's cpu_baseline leg
#   oracle/_ref/refcheck/  the reference's own unittest files next to an import shim (`datasketch` -> datasketch_b200),
#                          run by tests/test_reference_own_tests_{cpu,gpu}.py
# Nothing under oracle/_ref/ is committed; a built tree carries it to wherever the tests and the bench run.
#   bash oracle/stage_reference.sh [REFERENCE_CHECKOUT]      (default: $DATASKETCH_REF, else /root/reference)
# The reference's build backend (hatchling) may be missing offline, and the package is pure Python, so a wheel is
# zipped by hand from a scratch copy (nothing is written to the checkout) and pip installs THAT wheel with
# --no-index --no-deps --target.
set -euo pipefail
REPO="$(cd "$(dirname "$0")/.." && pwd)"
REF=${1:-${DATASKETCH_REF:-/root/reference}}
[ -d "$REF/datasketch" ] && [ -d "$REF/test" ] || { echo "no reference checkout at $REF"; exit 1; }
OUT="$REPO/oracle/_ref"
TMP=$(mktemp -d)
trap 'rm -rf "$TMP"' EXIT

# ---- the package ----
VER=$(sed -n 's/^version = "\(.*\)"/\1/p' "$REF/pyproject.toml" | head -1)
mkdir -p "$TMP/w" && cp -r "$REF/datasketch" "$TMP/w/datasketch"
find "$TMP/w" -name __pycache__ -prune -exec rm -rf {} +
DI="$TMP/w/datasketch-$VER.dist-info"; mkdir -p "$DI"
printf 'Metadata-Version: 2.1\nName: datasketch\nVersion: %s\nRequires-Dist: numpy>=1.11\nRequires-Dist: scipy>=1.0.0\n' "$VER" > "$DI/METADATA"
printf 'Wheel-Version: 1.0\nGenerator: oracle/stage_reference.sh\nRoot-Is-Purelib: true\nTag: py3-none-any\n' > "$DI/WHEEL"
( cd "$TMP/w" && find . -type f ! -name RECORD | sed 's#^\./##' | awk '{print $0",,"}' > "$DI/RECORD" && echo "datasketch-$VER.dist-info/RECORD,," >> "$DI/RECORD" )
( cd "$TMP/w" && python -m zipfile -c "$TMP/datasketch-$VER-py3-none-any.whl" datasketch "datasketch-$VER.dist-info" )
rm -rf "$OUT/site"
python -m pip install -q --no-index --no-deps --target "$OUT/site" "$TMP/datasketch-$VER-py3-none-any.whl"
python - <<PY
import sys; sys.path.insert(0, "$OUT/site")
import datasketch; m = datasketch.MinHash(4, 1); m.update(b"Hello")
assert m.hashvalues.tolist() == [734825475, 960773806, 359816889, 342714745]
PY

# ---- the reference's own unittest files + the import shim ----
S="$OUT/refcheck"
rm -rf "$S" && mkdir -p "$S/datasketch" "$S/test"
for f in __init__.py utils.py test_minhash.py test_lean_minhash.py test_weighted_minhash.py test_lsh.py test_lshforest.py test_lshensemble.py test_lshbloom.py; do
  cp "$REF/test/$f" "$S/test/"
done
cat > "$S/datasketch/__init__.py" <<'PY'
from datasketch_b200 import *  # noqa
from datasketch_b200 import (MinHash, LeanMinHash, MinHashLSH, MinHashLSHForest, MinHashLSHEnsemble, WeightedMinHash,
                             WeightedMinHashGenerator, bBitMinHash, MinHashLSHBloom)
PY
for m in minhash lean_minhash weighted_minhash lsh lshforest lshensemble lsh_bloom b_bit_minhash hashfunc; do
cat > "$S/datasketch/$m.py" <<PY
import datasketch_b200.$m as _m
from datasketch_b200.$m import *  # noqa
globals().update({k: getattr(_m, k) for k in dir(_m) if not k.startswith("__")})
PY
done
cat > "$S/mockredis.py" <<'PY'
import unittest
def mock_redis_client(**kwargs):
    raise unittest.SkipTest("redis storage is out of scope")
mock_strict_redis_client = mock_redis_client
PY
echo "staged: oracle/_ref/site (datasketch $VER), oracle/_ref/refcheck"
