"""The kernels at their limits on the GPU: num_perm at and across the tile widths, the shared-memory budget and the API's
bounds; database and query counts at tile edges; grids large enough that the grid-stride loops wrap; inputs that push
the top-k prefilter's queue to its capacity.  Every case is compared exactly with a plain reference of the same
operation: brute-force numpy counts for top-k, the C oracle for Jaccard pairs and signatures, the numpy restatement of
the reference for Weighted MinHash (bit-exact with the host logarithm), the dict LSH and the host LSH Forest class.
The grid sizes named below are those of a B200 (148 SMs); the tests read the SM count and check the wrap is reached."""
import numpy as np
import pytest

from oracle import oracle_clib as oc
from oracle import oracle_np as o

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dsk():
    import datasketch_b200
    return datasketch_b200


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- all-pairs top-k (jaccard_kernels.cu) ------------------------------------------------------------------------------
def _check_topk(dsk, q, db, topk, self_base):
    """Both kernels (default = fingerprint prefilter where it applies, and the exact kernel) against brute force."""
    k = q.shape[1]
    wc, wi = o.jaccard_topk(q, db, topk, self_base)
    for pf in (True, False):
        cnt, idx = dsk.codec.jaccard_topk(q, db, topk=topk, self_base=self_base, to_host=False, prefilter=pf)
        cnt, idx = cnt.cpu().numpy(), idx.cpu().numpy()
        assert np.array_equal(idx, wi), dict(k=k, n=len(db), nq=len(q), topk=topk, self_base=self_base, prefilter=pf)
        assert np.array_equal(cnt.astype(np.int64), wc), dict(k=k, n=len(db), nq=len(q), prefilter=pf)


# (n, nq, topk, self_base): database counts around the 4-tile threshold of the prefilter (512) and several tiles deep,
# query counts around one 64-row query tile, self exclusion off / from row 0 / from a row in the middle of a tile
_TOPK_SHAPES = [(511, 65, 32, -1), (512, 64, 1, 0), (513, 63, 32, 70), (5000, 200, 32, 1037), (5000, 1, 1, -1),
                (513, 200, 1, -1)]


@pytest.mark.parametrize("k", [1, 31, 32, 33, 100, 480, 481, 512, 513, 736, 737, 1024, 4096])
def test_topk_num_perm_range_vs_brute_force(dsk, k):
    """num_perm across the prefilter's applicability (32 <= K <= 480: its bit planes fit a block's 227 KB of shared
    memory), the old whole-query-tile limit of the exact kernel (736), and the API's maximum (4096)."""
    rs = np.random.RandomState(k)
    for n, nq, topk, self_base in _TOPK_SHAPES:
        if k >= 1024 and nq == 200:
            nq = 65                                     # keeps the brute force small; the query tiles still wrap once
        db = rs.randint(0, 3, size=(n, k)).astype(np.uint32)          # low entropy: heavy ties
        db[rs.randint(0, n, n // 20)] = db[rs.randint(0, n, n // 20)]    # exact duplicates
        if self_base >= 0:
            q = np.ascontiguousarray(db[self_base:self_base + nq])
        else:
            q = rs.randint(0, 3, size=(nq, k)).astype(np.uint32)
            q[: nq // 3] = db[rs.randint(0, n, nq // 3)]
        _check_topk(dsk, q, db, topk, self_base)


@pytest.mark.parametrize("k", [64, 100, 480])
def test_topk_prefilter_queue_full(dsk, k):
    """Every value is a base value XOR 0x00010001 or not: such values differ but share their 16-bit fingerprint
    (v ^ v >> 16), so every (query, row) pair has an upper bound of K and all 8192 pairs of a tile enter the queue.
    The database keeps only a few positions truly equal to the queries, so the true counts are small and varied."""
    rs = np.random.RandomState(k + 1)
    n, nq = 700, 130
    base = rs.randint(0, 1 << 32, size=k, dtype=np.uint64).astype(np.uint32)
    flip = np.uint32(0x00010001)
    q = np.tile(base, (nq, 1))
    q[rs.uniform(size=q.shape) < 0.05] ^= flip
    db = np.tile(base ^ flip, (n, 1))
    eq = rs.uniform(size=db.shape) < rs.uniform(0, 0.2, size=(n, 1))
    db[eq] = np.tile(base, (n, 1))[eq]
    fp = lambda v: (v ^ (v >> 16)) & 0xFFFF                          # noqa: E731
    assert (fp(q) == fp(base)[None, :]).all() and (fp(db) == fp(base)[None, :]).all()
    for topk, self_base in ((32, -1), (5, -1)):
        _check_topk(dsk, q, db, topk, self_base)
    q2 = np.ascontiguousarray(db[100:100 + nq])
    _check_topk(dsk, q2, db, 32, 100)


def test_topk_grid_stride_wraps(dsk):
    """30 000 queries = 469 query tiles: more than the prefilter's grid (2 CTAs per SM, wrapping at query row 18 944 on a
    B200) and the exact kernel's (3 per SM, wrapping at 28 416), so both re-initialise their per-tile state on a wrap.
    The two kernels must agree on every row, and every row is checked against brute force."""
    rs = np.random.RandomState(30)
    k, n, nq = 32, 600, 30_000
    assert nq > 3 * _sm_count() * 64
    db = rs.randint(0, 4, size=(n, k)).astype(np.uint32)
    q = rs.randint(0, 4, size=(nq, k)).astype(np.uint32)
    q[::7] = db[rs.randint(0, n, len(q[::7]))]
    res = {}
    for pf in (True, False):
        cnt, idx = dsk.codec.jaccard_topk(q, db, topk=32, to_host=False, prefilter=pf)
        res[pf] = (cnt.cpu().numpy().astype(np.int64), idx.cpu().numpy())
    assert np.array_equal(res[True][0], res[False][0]) and np.array_equal(res[True][1], res[False][1])
    wc, wi = o.jaccard_topk(q, db, 32)
    for lo, hi in ((0, nq), (18_880, 19_008), (28_352, 28_480), (29_952, nq)):   # whole matrix, then the wrap points
        assert np.array_equal(res[True][1][lo:hi], wi[lo:hi]) and np.array_equal(res[True][0][lo:hi], wc[lo:hi]), (lo, hi)


def test_topk_api_limits(dsk):
    q = np.zeros((2, 4097), dtype=np.uint32)
    with pytest.raises(ValueError):
        dsk.codec.jaccard_topk(q, q, topk=1)            # num_perm > 4096
    q = np.zeros((2, 64), dtype=np.uint32)
    with pytest.raises(ValueError):
        dsk.codec.jaccard_topk(q, q, topk=33)           # topk > 32


# ---- Jaccard pairs: the scalar path (num_perm not a multiple of 4) ---------------------------------------------------
@pytest.mark.parametrize("k", [1, 3, 5, 127, 129, 1023])
def test_jaccard_pairs_scalar_path(dsk, k):
    rs = np.random.RandomState(k)
    n, m = 3000, 20_000
    sig = rs.randint(0, 3, size=(n, k)).astype(np.uint32)
    ia, ib = rs.randint(0, n, size=m), rs.randint(0, n, size=m)
    ia[:50] = ib[:50]                                   # a row with itself: count = num_perm
    ia[50], ib[50] = n - 1, n - 1
    got = dsk.codec.jaccard_pairs(sig, ia, ib)
    cnt = oc.jaccard_pairs_u32(sig, ia, ib)
    assert np.array_equal(cnt[:51], np.full(51, k))
    assert np.array_equal(got, cnt.astype(np.float64) / k)


# ---- Weighted MinHash (wmh_kernels.cu) ---------------------------------------------------------------------------------
def _wmh_weights(rs, n, dim, negatives):
    """Zeros, subnormals (1e-40), values next to FLT_MAX (3e38), ordinary values, negatives (NaN after the logarithm, skipped
    by the reference's nanargmin) when asked, and a row whose only nonzero weight is the last dimension."""
    X = rs.uniform(0, 10, size=(n, dim)).astype(np.float32)
    u = rs.uniform(size=(n, dim))
    X[u < 0.3] = 0
    X[(u >= 0.3) & (u < 0.35)] = np.float32(1e-40)
    X[(u >= 0.35) & (u < 0.4)] = np.float32(3e38)
    if negatives:
        X[(u >= 0.4) & (u < 0.5)] *= -1
    X[:, 0] = np.where(X[:, 0] > 0, X[:, 0], np.float32(0.5))        # every row keeps a positive weight
    if n > 1:
        X[n - 1] = 0
        X[n - 1, dim - 1] = np.float32(2.5)
    return X


@pytest.mark.parametrize("ss", [1, 127, 128, 129, 257])
@pytest.mark.parametrize("dim", [1, 3, 5, 255, 256, 257, 1029])
def test_wmh_shapes_vs_oracle_exact(dsk, dim, ss):
    """Sample counts across the 128-thread blockIdx.y slices, dimension counts that leave a tail after the 4-way unroll
    and cross several 256-wide tiles, vector counts around the 8-vector group.  With the host logarithm every step is
    the reference's float32 op in the reference's order: zero mismatches."""
    rs = np.random.RandomState(dim * 1000 + ss)
    gen = dsk.WeightedMinHashGenerator(dim, ss, 7)
    par = (gen.rs, gen.ln_cs, gen.betas)
    for n in (1, 8, 9):
        X = _wmh_weights(rs, n, dim, negatives=True)
        with np.errstate(invalid="ignore", divide="ignore"):
            want = np.stack([o.wmh_minhash(v, *par) for v in X])
        got = gen.minhash_batch(X)
        assert np.array_equal(got, want), (dim, ss, n)
        # minhash_many: the reference's argmin does not skip NaN, so its input has no negative weights
        Xm = np.abs(X)
        Xm[0] = 0                                       # an all-zero row -> None
        with np.errstate(invalid="ignore", divide="ignore"):
            want_m = o.wmh_minhash_many(Xm, *par)
        got_m = gen.minhash_many(Xm)
        assert [m is None for m in got_m] == [w is None for w in want_m]
        for g, w in zip(got_m, want_m):
            if w is not None:
                assert np.array_equal(g.hashvalues, w), (dim, ss, n)


def test_wmh_grid_stride_wraps(dsk):
    """10 000 vectors = 1250 groups of 8: more than the grid's 8 CTAs per SM (the wrap starts at vector 9472 on a B200)."""
    rs = np.random.RandomState(10)
    dim, ss, n = 5, 129, 10_000
    assert n > _sm_count() * 8 * 8
    gen = dsk.WeightedMinHashGenerator(dim, ss, 3)
    par = (gen.rs, gen.ln_cs, gen.betas)
    X = _wmh_weights(rs, n, dim, negatives=True)
    got = gen.minhash_batch(X)
    wrap = _sm_count() * 8 * 8
    rows = sorted(set(range(0, 16)) | set(range(0, n, 97)) | set(range(wrap - 16, wrap + 16)) | set(range(n - 16, n)))
    with np.errstate(invalid="ignore", divide="ignore"):
        for i in rows:
            assert np.array_equal(got[i], o.wmh_minhash(X[i], *par)), i


# ---- signature kernel: K slices, piece mode, running state, u64 tokens -----------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 31, 33, 65, 129, 257, 512, 1024, 4096, 16384])
def test_signature_kernel_num_perm_range(dsk, k):
    """num_perm 512 / 1024 / 4096 / 16384 are 2 / 4 / 16 / 64 K-slices of the signature kernel.  tokens x K stays near
    10^8 so the C oracle stays fast; one document is longer than 4096 tokens (cut into pieces on the device)."""
    import torch
    rs = np.random.RandomState(k)
    budget = min(200_000, 100_000_000 // k)
    lens = [5000, 0, 1, 17, 300]
    while sum(lens) < budget:
        lens.append(int(rs.randint(0, 400)))
    lens = np.array(lens, dtype=np.int64)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    T, n = int(off[-1]), len(lens)
    tok = rs.randint(0, 1 << 32, size=T, dtype=np.uint64).astype(np.uint32)
    tok[100:2000] = tok[2000:3900]                      # repeats inside the long document
    P = o.init_permutations(k, 2)
    want = oc.minhash_bulk_u32tok(tok, off, P)
    assert np.array_equal(dsk.engine.bulk_signatures(tok, off, P), want)
    d_tok = torch.from_numpy(np.concatenate([tok, np.zeros(4, np.uint32)]).view(np.int32)).cuda()[:T]
    d_off = torch.from_numpy(off).cuda()
    got = dsk.engine.bulk_signatures_device(d_tok, d_off, T, P).cpu().numpy().view(np.uint32)
    assert np.array_equal(got, want)
    # running state: one row broadcast (host entry), one row per document (device entry, u64 output)
    row = rs.randint(0, 1 << 32, size=k, dtype=np.uint64)
    got = dsk.engine.bulk_signatures(tok, off, P, init=row, out_u64=True)
    assert np.array_equal(got, np.minimum(want.astype(np.uint64), row[None, :]))
    init = rs.randint(0, 1 << 32, size=(n, k), dtype=np.uint64)
    d_out = torch.empty((n, k), dtype=torch.int64, device="cuda")
    dsk.engine.bulk_signatures_device(d_tok, d_off, T, P, d_out=d_out, d_init=torch.from_numpy(init.view(np.int64)).cuda(),
                                      init_stride=k)
    assert np.array_equal(d_out.cpu().numpy().view(np.uint64), np.minimum(want.astype(np.uint64), init))
    if k in (33, 512, 4096):                            # 64-bit tokens
        tok64 = (rs.randint(0, 1 << 32, size=T, dtype=np.uint64) << np.uint64(32)) | tok.astype(np.uint64)
        want64 = oc.minhash_bulk_u64tok(tok64, off, P)
        assert np.array_equal(dsk.engine.bulk_signatures(tok64, off, P), want64)
        d_tok64 = torch.from_numpy(tok64.view(np.int64)).cuda()
        assert np.array_equal(dsk.engine.bulk_signatures_device(d_tok64, d_off, T, P).cpu().numpy().view(np.uint32), want64)


def test_signature_kernel_num_perm_above_limit(dsk):
    P = o.init_permutations(16385, 1)
    with pytest.raises(ValueError):
        dsk.engine.bulk_signatures(np.arange(10, dtype=np.uint32), np.array([0, 10]), P)


# ---- device LSH index and forest -----------------------------------------------------------------------------------
@pytest.mark.parametrize("params", [(2, 512), (4, 200)])
def test_gpu_lsh_wide_rows_vs_dict_oracle(dsk, params):
    """num_perm 1024 with few bands: a document's row (4 KB) forces lsh_insert_kernel to shrink its tile below 48 KB;
    (4, 200) leaves 224 positions unused.  The index is filled exactly to capacity in two inserts."""
    k = 1024
    b, r = params
    rs = np.random.RandomState(b)
    n = 1500
    sig = rs.randint(0, 1 << 32, size=(n, k), dtype=np.uint64).astype(np.uint32)
    src = rs.randint(0, n, 300)
    dst = rs.randint(0, n, 300)
    for s_, d_ in zip(src, dst):                        # rows sharing some bands (and not others) with an earlier row
        band = int(rs.randint(0, b))
        sig[d_, band * r:(band + 1) * r] = sig[s_, band * r:(band + 1) * r]
    sig[rs.randint(0, n, 50)] = sig[rs.randint(0, n, 50)]
    sig[7, b * r:] = sig[8, b * r:] + 1                 # unused tail positions differ, every band equal
    sig[7, :b * r] = sig[8, :b * r]
    ix = dsk.GpuLSH(num_perm=k, params=params, capacity=n)
    ix.insert(sig[:1000])
    ix.insert(sig[1000:])
    assert len(ix) == n
    with pytest.raises(ValueError):
        ix.insert(sig[:1])                              # full
    ref = o.DictLSH(k, b, r)
    for i, row in enumerate(sig):
        ref.insert(i, row.astype(np.uint64))
    q = np.concatenate([sig[::3], rs.randint(0, 1 << 32, size=(20, k), dtype=np.uint64).astype(np.uint32)])
    ptr, idx = ix.query(q)
    multi = 0
    for j in range(len(q)):
        got = sorted(idx[ptr[j]:ptr[j + 1]].tolist())
        assert got == sorted(ref.query(q[j].astype(np.uint64))), j
        multi += len(got) > 1
    assert multi > 20
    _, i8 = ix.query(sig[8:9])
    assert 7 in i8.tolist() and 8 in i8.tolist()
    empty = np.zeros((0, k), dtype=np.uint32)
    ix2 = dsk.GpuLSH(num_perm=k, params=params, capacity=10)
    ix2.insert(empty)
    assert len(ix2) == 0
    ptr, idx = ix2.query(sig[:3])
    assert ptr.tolist() == [0, 0, 0, 0] and len(idx) == 0
    ptr, idx = ix.query(empty)
    assert ptr.tolist() == [0] and len(idx) == 0


def test_gpu_forest_one_column_trees_and_large_topk(dsk):
    """l = 64 trees of k = 1 column at num_perm 64 (the query kernel's lanes take the 64 trees in two rounds) and topk
    up to 1024, against the host MinHashLSHForest (pinned to the reference's fixtures in tests/test_lshforest.py)."""
    rs = np.random.RandomState(64)
    K, l, n = 64, 64, 3000
    sig = rs.randint(0, 40, size=(n, K)).astype(np.uint32)
    sig[rs.randint(0, n, 200)] = sig[rs.randint(0, n, 200)]
    f = dsk.MinHashLSHForest(num_perm=K, l=l)
    for i, row in enumerate(sig):
        f.add(i, dsk.LeanMinHash(seed=1, hashvalues=row.astype(np.uint64)))
    f.index()
    dev = dsk.GpuLSHForest(num_perm=K, l=l)
    dev.add(sig)
    dev.index()
    q = np.concatenate([sig[:30], rs.randint(0, 40, size=(10, K)).astype(np.uint32)])
    for topk in (1, 64, 1024):
        res = dev.query(q, topk)
        for j, row in enumerate(q):
            want = sorted(f.query(dsk.LeanMinHash(seed=1, hashvalues=row.astype(np.uint64)), topk))
            assert sorted(int(x) for x in res[j] if x >= 0) == want, (topk, j)
