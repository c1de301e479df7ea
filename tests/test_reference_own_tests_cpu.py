"""The reference's OWN unittest files, run against datasketch_b200 on the CPU.

The files are staged by ``oracle/stage_reference.sh`` (run by ``build()`` where a reference checkout is readable) into
the git-ignored ``oracle/_ref/refcheck/`` next to an import shim (``datasketch`` -> ``datasketch_b200``); without them the
test is skipped (``tests/test_api_behaviour.py`` is the self-contained comparison with the reference).  They run in a
subprocess with the emulated library (``tests/emu/emu_capi.cpp``) swapped in for ``libdsk_b200.so``.  Covered here: the
tests whose code path needs only host buffers (MinHash / LeanMinHash / bBitMinHash / MinHashLSH / MinHashLSHForest on
MinHash signatures); the Weighted MinHash and ensemble / LSHBloom tests need torch CUDA tensors and run in the GPU
variant of this check (``tests/test_reference_own_tests_gpu.py``, part of ``pytest -m gpu``).
"""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGE = os.path.join(ROOT, "oracle", "_ref", "refcheck")

pytestmark = pytest.mark.skipif(not os.path.isdir(os.path.join(STAGE, "test")) or shutil.which("g++") is None,
                                reason="needs the reference's test files staged in oracle/_ref/refcheck/ "
                                       "(oracle/stage_reference.sh) and g++")

_BOOT = '''
import ctypes, os, sys
sys.path[:0] = [{stage!r}, {root!r}]
from datasketch_b200 import _native as nv
lib = ctypes.CDLL(os.path.join({root!r}, "tests", "emu", "_build", "libdsk_emu.so"))
for name, (res, args) in nv.SIGNATURES.items():
    fn = getattr(lib, name)
    fn.restype, fn.argtypes = res, args
nv._perm_cache.clear()
nv._lib = lib                                   # test-only: the emulated library stands in for libdsk_b200.so
import pytest
sys.exit(pytest.main(["-q", "-p", "no:cacheprovider", "-k", {select!r}] + {files!r}))
'''


def test_reference_unittests_pass_on_the_emulated_library(request):
    request.getfixturevalue("emu_lib")          # builds tests/emu/_build/libdsk_emu.so
    files = [os.path.join(STAGE, "test", f) for f in
             ("test_minhash.py", "test_lean_minhash.py", "test_lsh.py", "test_lshforest.py")]
    # test_unpacking spends a minute in the host-side (b, r) optimiser (scipy quad); it runs in the GPU variant
    select = "not redis and not Weighted and not unpacking"
    code = _BOOT.format(stage=STAGE, root=ROOT, select=select, files=files)
    run = subprocess.run([sys.executable, "-c", code], cwd=STAGE, capture_output=True, text=True, timeout=1200)
    tail = (run.stdout + run.stderr)[-3000:]
    assert run.returncode == 0, tail
    assert " passed" in tail and "failed" not in tail, tail
    assert int(tail.split(" passed")[0].split()[-1]) >= 45, tail
