"""The reference's OWN unittest files, run against datasketch_b200 on the GPU -- the drop-in gate.

``oracle/stage_reference.sh`` (run by ``build()`` where a reference checkout is readable) stages ekzhu/datasketch's
``test/test_minhash.py``, ``test_lean_minhash.py``, ``test_weighted_minhash.py``, ``test_lsh.py``, ``test_lshforest.py``,
``test_lshensemble.py`` and ``test_lshbloom.py`` next to an import shim (``datasketch`` -> ``datasketch_b200``) in the
git-ignored ``oracle/_ref/refcheck/``, which a built tree carries along.  Here the files run unchanged in a subprocess
against the real library.  Deselected: the Redis-backed cases (storage backends are out of scope; the shim's
``mockredis`` raises SkipTest).  Without the staged files the test is SKIPPED with that reason -- it never passes
vacuously; ``tests/test_api_behaviour.py`` is the self-contained comparison with the reference.
"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGE = os.path.join(ROOT, "oracle", "_ref", "refcheck")
FILES = ["test_minhash.py", "test_lean_minhash.py", "test_weighted_minhash.py", "test_lsh.py", "test_lshforest.py",
         "test_lshensemble.py", "test_lshbloom.py"]


@pytest.mark.gpu
def test_reference_unittests_pass_on_the_gpu(tmp_path):
    if not os.path.isdir(os.path.join(STAGE, "test")):
        pytest.skip("the reference's test files are not staged (oracle/_ref/refcheck/ absent: build() stages them "
                    "where a reference checkout is readable, see oracle/stage_reference.sh)")
    files = [os.path.join(STAGE, "test", f) for f in FILES if os.path.exists(os.path.join(STAGE, "test", f))]
    assert len(files) == len(FILES), files
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([STAGE, ROOT, os.environ.get("PYTHONPATH", "")]))
    run = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-k", "not redis"] + files,
                         cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=1500)
    tail = (run.stdout + run.stderr)[-4000:]
    assert run.returncode == 0, tail
    assert " passed" in tail and " failed" not in tail, tail
    assert int(tail.split(" passed")[0].split()[-1]) >= 75, tail
