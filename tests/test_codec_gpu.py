"""GPU parity: LeanMinHash record codec and LSH band keys vs reference-made fixtures and the oracle."""
import pickle

import numpy as np
import pytest

from oracle import oracle_clib as oc
from oracle import oracle_np as o

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dsk():
    import datasketch_b200
    return datasketch_b200


def test_lean_pack_golden_batch(dsk, golden):
    g = golden("lean")
    rec = dsk.codec.lean_pack(g["batch_sig"], seed=9).cpu().numpy()
    assert rec.shape == (16, 12 + 4 * 128) and np.array_equal(rec, g["batch_recs"])
    back = dsk.codec.lean_unpack(rec, 128, 9).cpu().numpy().view(np.uint32)
    assert np.array_equal(back, g["batch_sig"])
    with pytest.raises(ValueError):
        dsk.codec.lean_unpack(rec, 128, 10)  # wrong seed in header


@pytest.mark.parametrize("k", [4, 10, 100, 128, 256, 1000])
@pytest.mark.parametrize("bo", ["@", "<", ">", "!"])
def test_lean_pack_all_byteorders_vs_struct(dsk, k, bo):
    rs = np.random.RandomState(k)
    n = 37 if k > 100 else 301
    sig = rs.randint(0, 2 ** 32, size=(n, k), dtype=np.uint64).astype(np.uint32)
    seed = -123456789012345 if k % 2 else 7
    rec = dsk.codec.lean_pack(sig, seed=seed, byteorder=bo).cpu().numpy()
    for i in (0, n // 2, n - 1):
        assert rec[i].tobytes() == o.lean_serialize(seed, sig[i].astype(np.uint64), bo)
    back = dsk.codec.lean_unpack(rec, k, seed, byteorder=bo).cpu().numpy().view(np.uint32)
    assert np.array_equal(back, sig)
    back64 = dsk.codec.lean_unpack(rec, k, seed, byteorder=bo, out_u64=True).cpu().numpy().view(np.uint64)
    assert np.array_equal(back64, sig.astype(np.uint64))
    # u64 input matrix (the reference's in-memory dtype) packs to the same bytes
    rec64 = dsk.codec.lean_pack(sig.astype(np.uint64), seed=seed, byteorder=bo).cpu().numpy()
    assert np.array_equal(rec64, rec)


def test_lean_pack_large_roundtrip_and_checksum(dsk):
    # size-independent properties at a large size: unpack(pack(x)) == x; header words constant
    import torch
    n, k = 200_003, 128
    sig = torch.randint(-2 ** 31, 2 ** 31 - 1, (n, k), dtype=torch.int32, device="cuda")
    rec = dsk.codec.lean_pack(sig, seed=1)
    assert torch.equal(dsk.codec.lean_unpack(rec, k, 1), sig)
    words = rec.view(torch.int32).view(n, k + 3)
    assert bool((words[:, 0] == 1).all()) and bool((words[:, 1] == 0).all()) and bool((words[:, 2] == k).all())
    assert torch.equal(words[:, 3:], sig)


def test_lean_object_api_matches_reference_bytes(dsk, golden):
    g = golden("lean")
    lm = dsk.LeanMinHash(seed=int(g["seed"]), hashvalues=g["hashvalues"])
    for bo, nm in {"@": "native", "=": "std", "<": "le", ">": "be", "!": "net"}.items():
        assert lm.bytesize(bo) == int(g[f"size_{nm}"])
        buf = bytearray(lm.bytesize(bo))
        lm.serialize(buf, bo)
        assert np.array_equal(np.frombuffer(bytes(buf), np.uint8), g[f"buf_{nm}"])
        back = dsk.LeanMinHash.deserialize(buf, bo)
        assert back.seed == lm.seed and np.array_equal(back.hashvalues, lm.hashvalues) and back == lm
    assert bytes(lm.__getstate__()) == g["getstate"].tobytes()
    assert hash(lm) == int(g["pyhash"])
    p = pickle.loads(pickle.dumps(lm))
    assert p == lm and p.hashvalues.dtype == np.uint64
    with pytest.raises(TypeError):
        lm.update(b"x")
    with pytest.raises(ValueError):
        lm.serialize(bytearray(3))
    m = dsk.MinHash(10, 1, hashfunc=int)
    m.update(123)
    assert dsk.LeanMinHash(m) == lm and dsk.LeanMinHash(m).jaccard(lm) == 1.0
    c = lm.copy()
    assert c == lm and c.hashvalues is not lm.hashvalues
    assert dsk.LeanMinHash.union(lm, dsk.LeanMinHash(dsk.MinHash(10, 1))) == lm


@pytest.mark.parametrize("k,b,r", [(128, 9, 13), (128, 32, 4), (256, 17, 15), (16, 4, 4), (8, 4, 2)])
def test_band_keys_vs_oracle(dsk, k, b, r):
    rs = np.random.RandomState(b * r)
    sig = rs.randint(0, 2 ** 32, size=(211, k), dtype=np.uint64).astype(np.uint32)
    keys = dsk.codec.band_keys(sig, b, r).cpu().numpy()
    assert keys.shape == (211, b, 8 * r)
    assert np.array_equal(keys, oc.band_keys_be(sig, b, r))
    for i in (0, 100, 210):
        want = o.lsh_band_keys(sig[i].astype(np.uint64), b, r)
        assert [keys[i, j].tobytes() for j in range(b)] == want
    with pytest.raises(ValueError):
        dsk.codec.band_keys(sig, b + k, r)


def test_band_keys_golden_and_fingerprints(dsk, golden):
    g = golden("lsh")
    b, r = [int(x) for x in g["b_r"]]
    sig = g["sig"]
    keys = dsk.codec.band_keys(sig, b, r).cpu().numpy()
    assert np.array_equal(keys[0], g["keys_doc0"])
    fp = dsk.codec.band_fingerprints(sig, b, r).cpu().numpy().view(np.uint64)
    # fingerprints agree exactly where (and essentially only where) the band keys agree
    for j in range(b):
        kj = [keys[i, j].tobytes() for i in range(len(sig))]
        same_key = np.array([[a == c for c in kj[:60]] for a in kj[:60]])
        same_fp = fp[:60, j][:, None] == fp[:60, j][None, :]
        assert np.array_equal(same_key, same_fp)
    assert len(np.unique(fp)) > 0.5 * fp.size


@pytest.mark.parametrize("k", [128, 100, 256, 4])
def test_jaccard_pairs_vs_oracle(dsk, k):
    rs = np.random.RandomState(k)
    n, m = 5000, 20000
    sig = rs.randint(0, 4, size=(n, k)).astype(np.uint32)     # low entropy: many equal positions
    ia, ib = rs.randint(0, n, size=m), rs.randint(0, n, size=m)
    ia[:10] = ib[:10]                                          # identical rows -> 1.0
    got = dsk.codec.jaccard_pairs(sig, ia, ib)
    want = oc.jaccard_pairs_u32(sig, ia, ib).astype(np.float64) / k
    assert got.dtype == np.float64 and np.array_equal(got, want) and (got[:10] == 1.0).all()
    for p in range(5):
        assert got[p] == o.jaccard(sig[ia[p]].astype(np.uint64), sig[ib[p]].astype(np.uint64))
    with pytest.raises(IndexError):
        dsk.codec.jaccard_pairs(sig, [0, n], [1, 2])


def test_jaccard_pairs_matches_golden_objects(dsk, golden):
    g = golden("minhash")
    sig = np.stack([g["j_m1"], g["j_m2"]]).astype(np.uint32)
    assert dsk.codec.jaccard_pairs(sig, [0], [1])[0] == float(g["j_jaccard"])


@pytest.mark.parametrize("k,n,nq,topk,self_base", [(128, 1000, 150, 10, 0), (100, 333, 70, 5, -1), (128, 7, 7, 10, 0),
                                                    (64, 2000, 65, 32, 500), (256, 300, 10, 1, -1)])
def test_jaccard_topk_vs_oracle(dsk, k, n, nq, topk, self_base):
    rs = np.random.RandomState(n + k)
    db = rs.randint(0, 3, size=(n, k)).astype(np.uint32)       # low entropy: many ties, large counts
    db[rs.randint(0, n, 20)] = db[rs.randint(0, n, 20)]
    if self_base >= 0:
        q = db[self_base:self_base + nq].copy()
        nq = len(q)
    else:
        q = rs.randint(0, 3, size=(nq, k)).astype(np.uint32)
    jac, idx = dsk.codec.jaccard_topk(q, db, topk=topk, self_base=self_base)
    wc, wi = o.jaccard_topk(q, db, topk, self_base)
    assert np.array_equal(idx, wi)
    assert np.array_equal(jac, np.where(wc >= 0, wc, 0) / float(k))


def test_jaccard_topk_random_signatures_finds_planted_pairs(dsk):
    # C5-shaped data, scaled: uniformly random signatures (all counts 0 -> ties by index) with planted near-duplicates
    rs = np.random.RandomState(5)
    n, k = 20_000, 128
    db = rs.randint(0, 2 ** 32, size=(n, k), dtype=np.uint64).astype(np.uint32)
    for i in range(0, 2000, 2):
        db[i + 1] = db[i]
        db[i + 1, rs.choice(k, 10, replace=False)] = 7
    q = db[:512]
    jac, idx = dsk.codec.jaccard_topk(q, db, topk=10, self_base=0)
    wc, wi = o.jaccard_topk(q[:64], db, 10, 0)
    assert np.array_equal(idx[:64], wi)
    assert all(idx[i, 0] == i + 1 for i in range(0, 512, 2)) and all(idx[i, 0] == i - 1 for i in range(1, 512, 2))
    assert (jac[:, 0] >= 118 / 128).all() and (jac[:, 1] < 0.1).all()


def test_sharded_topk_single_process_equals_kernel(dsk):
    """world size 1: distributed.sharded_jaccard_topk is the plain kernel with self_base = 0."""
    rs = np.random.RandomState(3)
    sig = rs.randint(0, 4, size=(500, 64)).astype(np.uint32)
    import torch
    d = torch.from_numpy(sig.view(np.int32)).cuda()
    cnt, idx = dsk.distributed.sharded_jaccard_topk(d, topk=7)
    wc, wi = o.jaccard_topk(sig, sig, 7, 0)
    assert np.array_equal(idx.cpu().numpy(), wi) and np.array_equal(cnt.cpu().numpy(), wc)
    full, base, counts = dsk.distributed.gather_signature_blocks(d)
    assert full is d and base == 0 and counts == [500]
