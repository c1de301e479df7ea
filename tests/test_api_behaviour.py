"""datasketch_b200 behaves as the reference does through the public API: the scenarios of oracle/api_scenarios.py
(ordinary use and misuse of MinHash, LeanMinHash, MinHashLSH, MinHashLSHForest) against what the unmodified reference
returned or raised in each of them (tests/golden/api_behaviour.json, written by oracle/gen_api_golden.py).  On the CPU
the emulated library (tests/emu/emu_capi.cpp) stands in for libdsk_b200.so; with -m gpu the real library runs."""
import json
import math
import os
import shutil

import pytest

from oracle.api_scenarios import SCENARIOS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "tests", "golden", "api_behaviour.json")) as _f:
    WANT = json.load(_f)


def _same(got, want, path):
    if isinstance(want, float) and isinstance(got, float):
        assert math.isclose(got, want, rel_tol=1e-12, abs_tol=0.0), path
    elif isinstance(want, dict) and isinstance(got, dict):
        assert sorted(got) == sorted(want), (path, got, want)
        for k in want:
            _same(got[k], want[k], path + "." + k)
    elif isinstance(want, list) and isinstance(got, list):
        assert len(got) == len(want), (path, got, want)
        for i, (g, w) in enumerate(zip(got, want)):
            _same(g, w, "%s[%d]" % (path, i))
    else:
        assert type(got) is type(want) and got == want, (path, got, want)


def _check(dsk, name):
    assert sorted(SCENARIOS) == sorted(WANT)
    got = json.loads(json.dumps(SCENARIOS[name](dsk)))
    _same(got, WANT[name], name)


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_api_behaviour_matches_reference_on_the_emulated_library(name, emu_lib, monkeypatch):
    import datasketch_b200 as dsk
    from datasketch_b200 import _native as nv
    nv._perm_cache.clear()
    monkeypatch.setattr(nv, "_lib", emu_lib)
    try:
        _check(dsk, name)
    finally:
        nv._perm_cache.clear()                # handles created on the emulated library die on it


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_api_behaviour_matches_reference_on_the_gpu(name):
    import datasketch_b200 as dsk
    _check(dsk, name)
