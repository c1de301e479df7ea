"""GPU parity: Weighted MinHash vs fixtures produced by the reference's own
WeightedMinHashGenerator.minhash (no value golden exists in the reference's tests)."""
import pickle

import numpy as np
import pytest

from oracle import oracle_np as o

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dsk():
    import datasketch_b200
    return datasketch_b200


def _explain_mismatch(v, rs, ln_cs, betas, got, want):
    """A (k,t) difference is only acceptable if it is a float near-tie: the oracle's ln_a at the two
    candidate indices differ by <= 1e-6 relative (north_star tolerance for the float step), or the
    floor argument sits within 1e-6 of an integer."""
    v = np.array(v, dtype=np.float32)
    v[v == 0] = np.nan
    vlog = np.log(v)
    bad = []
    for i in np.where((got != want).any(axis=1))[0]:
        t = np.floor(vlog / rs[i] + betas[i])
        ln_a = ln_cs[i] - (t - betas[i]) * rs[i] - rs[i]
        kg, kw = int(got[i, 0]), int(want[i, 0])
        near_tie = abs(float(ln_a[kg]) - float(ln_a[kw])) <= 1e-6 * max(1.0, abs(float(ln_a[kw])))
        arg = vlog[kw] / rs[i][kw] + betas[i][kw]
        near_int = abs(arg - np.round(arg)) <= 1e-6 * max(1.0, abs(arg))
        if not (near_tie or near_int):
            bad.append(int(i))
    return bad


@pytest.mark.parametrize("tag", ["small", "tiny", "c4"])
def test_wmh_matches_reference_fixture(dsk, golden, tag):
    g = golden("wmh")
    dim, ss, seed = [int(x) for x in g[f"{tag}_cfg"]]
    gen = dsk.WeightedMinHashGenerator(dim, ss, seed)
    rs, ln_cs, betas = o.wmh_params(dim, ss, seed)
    assert np.array_equal(gen.rs, rs) and np.array_equal(gen.ln_cs, ln_cs) and np.array_equal(gen.betas, betas)
    V, want = g[f"{tag}_v"], g[f"{tag}_out"]
    got = gen.minhash_batch(V)
    assert got.dtype == np.int64 and got.shape == want.shape
    # the logarithm is numpy's own (taken on the host), every later step is the reference's float32 op: exact
    assert np.array_equal(got, want), int((got != want).any(axis=2).sum())
    # object API, one vector at a time
    for u in (0, len(V) - 1):
        m = gen.minhash(V[u])
        assert isinstance(m, dsk.WeightedMinHash) and len(m) == ss and m.hashvalues.dtype == int
        assert np.array_equal(m.hashvalues, got[u])


def test_wmh_api_contract(dsk):
    # mirrors test/test_weighted_minhash.py:11-42 of the reference
    mg = dsk.WeightedMinHashGenerator(4, 10, 1)
    m = mg.minhash([1, 2, 3, 4])
    p = pickle.loads(pickle.dumps(m))
    assert p.seed == m.seed and np.array_equal(p.hashvalues, m.hashvalues)
    mg = dsk.WeightedMinHashGenerator(2, 4, 1)
    assert len(mg.rs) == 4 and len(mg.ln_cs) == 4 and len(mg.betas) == 4 and mg.seed == 1 and mg.sample_size == 4
    m = mg.minhash([1, 3])
    assert isinstance(m, dsk.WeightedMinHash) and len(m.hashvalues) == 4 and len(m) == 4
    assert m.hashvalues.dtype == int
    want = o.wmh_minhash([1, 3], *o.wmh_params(2, 4, 1))
    assert np.array_equal(m.hashvalues, want)
    mg = dsk.WeightedMinHashGenerator(3, 4, 1)
    v = np.array([1, 0, 3], dtype=np.float32)
    keep = v.copy()
    mg.minhash(v)
    np.testing.assert_array_equal(v, keep)
    with pytest.raises(ValueError):
        mg.minhash([0, 0, 0])
    with pytest.raises(ValueError):
        mg.minhash([1, 2])
    with pytest.raises(TypeError):
        mg.minhash(5)
    with pytest.raises(ValueError):
        mg.minhash_batch(np.array([[1, 2, 3], [0, 0, 0]], dtype=np.float32))
    a, b = mg.minhash([1, 2, 3]), mg.minhash([1, 2, 3])
    assert a == b and a.jaccard(b) == 1.0 and 0.0 <= a.jaccard(mg.minhash([3, 2, 1])) <= 1.0
    many = mg.minhash_many(np.array([[1, 2, 3], [3, 2, 1], [0, 0, 0]]))
    want_many = o.wmh_minhash_many(np.array([[1, 2, 3], [3, 2, 1], [0, 0, 0]]), *o.wmh_params(3, 4, 1))
    assert len(many) == 3 and many[2] is None and want_many[2] is None
    assert all(np.array_equal(many[i].hashvalues, want_many[i]) for i in range(2))
    with pytest.raises(TypeError):
        mg.minhash_many([[1, 2, 3]])               # reference: only numpy / scipy.sparse matrices
    with pytest.raises(ValueError):
        mg.minhash_many(np.array([1, 2, 3]))       # "Input must have two dimensions"
    with pytest.raises(ValueError):
        mg.minhash_many(np.ones((2, 4)))
    g2 = pickle.loads(pickle.dumps(mg))
    assert g2.minhash([1, 2, 3]) == a


def _random_batch(dsk):
    rs_ = np.random.RandomState(4)
    dim, ss = 300, 70        # neither a multiple of the tile / CTA sizes
    gen = dsk.WeightedMinHashGenerator(dim, ss, 11)
    V = rs_.uniform(0, 10, (27, dim)).astype(np.float32)
    V[:, ::7] = 0
    V[5] = np.floor(V[5])
    par = o.wmh_params(dim, ss, 11)
    return gen, V, par, np.stack([o.wmh_minhash(v, *par) for v in V])


def test_wmh_random_batch_vs_oracle(dsk):
    gen, V, par, want = _random_batch(dsk)
    got = gen.minhash_batch(V)
    # host logarithm: bit-identical by construction
    assert np.array_equal(got, want), int((got != want).any(axis=2).sum())


def test_wmh_device_log_differs_only_on_near_ties(dsk):
    gen, V, par, want = _random_batch(dsk)
    got = gen.minhash_batch(V, device_log=True)
    # the device's logarithm is within 1 ulp of numpy's: a (k, t) may differ only on a float near-tie
    for u in range(len(V)):
        if (got[u] != want[u]).any():
            assert _explain_mismatch(V[u], *par, got[u], want[u]) == []
    assert int((got != want).any(axis=2).sum()) <= 2


@pytest.mark.parametrize("tag", ["small", "tiny", "mid"])
def test_wmh_minhash_many_matches_reference_fixture(dsk, golden, tag):
    """minhash_many (dense and scipy.sparse input, all-zero rows -> None) against the outputs the
    reference produced for the same matrices (weighted_minhash.py:161-247)."""
    import scipy.sparse
    g = golden("wmh_many")
    dim, ss, seed = (int(x) for x in g[f"{tag}_cfg"])
    X, want, null = g[f"{tag}_X"], g[f"{tag}_out"], g[f"{tag}_null"]
    gen = dsk.WeightedMinHashGenerator(dim, ss, seed)
    for inp in (X, scipy.sparse.csr_matrix(X), scipy.sparse.coo_matrix(X)):
        got = gen.minhash_many(inp)
        assert isinstance(got, list) and len(got) == len(X)
        assert [m is None for m in got] == null.tolist()
        for i, m in enumerate(got):
            if m is not None:
                assert isinstance(m, dsk.WeightedMinHash) and m.seed == seed and m.hashvalues.dtype == int
                assert np.array_equal(m.hashvalues, want[i]), (tag, i)
