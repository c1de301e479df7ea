"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the datasketch hot path.

This file is the *oracle*: a CPU restatement of what the reference
(ekzhu/datasketch 1.10.0, mounted at /root/reference in the build container)
computes on the path named by BASELINE.json's north_star.  It exists so the GPU
box (which has no /root/reference) can check the CUDA path bit-for-bit.

Pinning status
    PINNED.  ``tests/test_oracle_golden.py`` checks every function here against
    fixtures under ``tests/golden/`` which were produced by importing the real
    reference in the build container (``oracle/gen_golden.py``), including the
    reference's own absolute golden vector (test/test_minhash.py:109-115).
    The weighted-MinHash path has no value golden in the reference's tests
    (test/test_weighted_minhash.py:29-35 checks dtype/len only); its fixtures are
    outputs of the reference's own ``WeightedMinHashGenerator.minhash`` run here.

The arithmetic physically lives in numpy (third-party; not under
/root/reference; pinned in the reference's uv.lock as numpy 2.0.2 / 2.2.6 /
2.3.4 by Python version).  This restatement therefore issues the *same numpy
ufuncs in the same order and dtypes* as the reference's call sites; each
function cites the reference file:line it follows.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module.
"""
from __future__ import annotations

import struct
from typing import Iterable, List, Sequence, Tuple

import numpy as np

# datasketch/minhash.py:30-32
MERSENNE_PRIME = np.uint64((1 << 61) - 1)
MAX_HASH = np.uint64((1 << 32) - 1)
HASH_RANGE = 1 << 32


# ----------------------------------------------------------------------------
# MinHash
# ----------------------------------------------------------------------------
def init_permutations(num_perm: int, seed: int) -> np.ndarray:
    """(2, num_perm) uint64; row 0 = a in [1,p), row 1 = b in [0,p).

    Follows datasketch/minhash.py:170-184: ONE RandomState(seed); for each
    permutation, in this interleaved order, ``randint(1, p)`` then
    ``randint(0, p)``, both dtype=uint64.
    """
    gen = np.random.RandomState(seed)
    pairs = []
    for _ in range(num_perm):
        a = gen.randint(1, MERSENNE_PRIME, dtype=np.uint64)
        b = gen.randint(0, MERSENNE_PRIME, dtype=np.uint64)
        pairs.append((a, b))
    return np.array(pairs, dtype=np.uint64).T


def init_hashvalues(num_perm: int) -> np.ndarray:
    """Empty signature = all 2^32-1 as uint64 (datasketch/minhash.py:167-168)."""
    return np.ones(num_perm, dtype=np.uint64) * MAX_HASH


def update_one(hashvalues: np.ndarray, hv: int, permutations: np.ndarray) -> np.ndarray:
    """One token (datasketch/minhash.py:221-224).

    ``hv`` is a Python int, so ``a * hv`` promotes exactly as in the reference
    (numpy uint64 array times Python int -> uint64 with wrap mod 2^64).
    """
    a, b = permutations
    with np.errstate(over="ignore"):
        phv = np.bitwise_and((a * hv + b) % MERSENNE_PRIME, MAX_HASH)
    return np.minimum(phv, hashvalues)


def update_batch(hashvalues: np.ndarray, hv_list: Sequence[int], permutations: np.ndarray) -> np.ndarray:
    """T tokens -> new signature (datasketch/minhash.py:262-266, 294-297).

    Empty batch is a no-op (:265-266).  The (T,1) x (K,) broadcast materialises
    the T x K uint64 temporary exactly as the reference does; the product wraps
    mod 2^64 *before* the ``% p`` (numpy uint64 semantics).
    """
    hv_list = list(hv_list)
    if not hv_list:
        return hashvalues
    a, b = permutations
    hv = np.array(hv_list, dtype=np.uint64, ndmin=2).T
    with np.errstate(over="ignore"):
        phv = (hv * a + b) % MERSENNE_PRIME
    phv = np.bitwise_and(phv, MAX_HASH)
    return np.minimum(hashvalues, phv.min(axis=0))


def bulk_signatures(docs: Iterable[Sequence[int]], num_perm: int, seed: int,
                    permutations: np.ndarray | None = None) -> np.ndarray:
    """[N, K] uint64 signature matrix of ``MinHash.bulk`` on integer token hashes.

    Follows datasketch/minhash.py:464-522: permutations are generated once
    (:518) and every document starts from the empty state (``m.copy()``, :520).
    """
    perms = init_permutations(num_perm, seed) if permutations is None else permutations
    base = init_hashvalues(num_perm)
    rows = [update_batch(base.copy(), d, perms) for d in docs]
    if not rows:
        return np.zeros((0, num_perm), dtype=np.uint64)
    return np.stack(rows)


def bulk_signatures_csr(tokens: np.ndarray, offsets: np.ndarray, num_perm: int, seed: int,
                        permutations: np.ndarray | None = None) -> np.ndarray:
    """Same as :func:`bulk_signatures` for a CSR batch (tokens[offsets[i]:offsets[i+1]])."""
    perms = init_permutations(num_perm, seed) if permutations is None else permutations
    n = len(offsets) - 1
    out = np.empty((n, num_perm), dtype=np.uint64)
    base = init_hashvalues(num_perm)
    a, b = perms
    for i in range(n):
        seg = tokens[int(offsets[i]):int(offsets[i + 1])]
        if len(seg) == 0:
            out[i] = base
            continue
        hv = seg.astype(np.uint64).reshape(-1, 1)
        with np.errstate(over="ignore"):
            phv = (hv * a + b) % MERSENNE_PRIME
        phv = np.bitwise_and(phv, MAX_HASH)
        out[i] = np.minimum(base, phv.min(axis=0))
    return out


def jaccard(hv1: np.ndarray, hv2: np.ndarray) -> float:
    """count_nonzero(h1 == h2) / K as a Python float (datasketch/minhash.py:324)."""
    return float(np.count_nonzero(hv1 == hv2)) / float(len(hv1))


def jaccard_topk(q: np.ndarray, db: np.ndarray, topk: int, self_base: int = -1) -> Tuple[np.ndarray, np.ndarray]:
    """Brute-force top-k by ``jaccard`` over two signature matrices, as counts of equal positions.

    Per query row: the ``topk`` database rows with the most equal positions, count descending then
    index ascending; ``self_base >= 0`` leaves database row ``self_base + i`` out of query i's list.
    Returns ``(count, index)``, both int64 [Q, topk], -1 where the database has fewer rows.  Counts
    are int64 sums of boolean compares, taken a few queries at a time to bound memory.
    """
    q, db = np.asarray(q), np.asarray(db)
    nq, n, k = len(q), len(db), q.shape[1]
    out_c = np.full((nq, topk), -1, np.int64)
    out_i = np.full((nq, topk), -1, np.int64)
    if nq == 0 or n == 0:
        return out_c, out_i
    excluded = np.int64((k + 1) * (n + 1))          # ranks after every real key
    step = max(1, (1 << 25) // max(1, n * k))
    for s in range(0, nq, step):
        blk = q[s:s + step]
        cnt = (blk[:, None, :] == db[None, :, :]).sum(axis=2, dtype=np.int64)
        key = (k - cnt) * (n + 1) + np.arange(n, dtype=np.int64)[None, :]      # count desc, then index asc
        if self_base >= 0:
            rows = self_base + np.arange(s, s + len(blk))
            hit = rows < n
            key[np.nonzero(hit)[0], rows[hit]] = excluded
        m = min(topk, n)
        order = np.argsort(key, axis=1, kind="stable")[:, :m]
        sel_key = np.take_along_axis(key, order, axis=1)
        keep = sel_key != excluded
        out_i[s:s + len(blk), :m] = np.where(keep, order, -1)
        out_c[s:s + len(blk), :m] = np.where(keep, np.take_along_axis(cnt, order, axis=1), -1)
    return out_c, out_i


def merge(hv1: np.ndarray, hv2: np.ndarray) -> np.ndarray:
    """Element-wise min (datasketch/minhash.py:359)."""
    return np.minimum(hv2, hv1)


def count(hashvalues: np.ndarray) -> float:
    """Cardinality estimate (datasketch/minhash.py:334-335)."""
    k = len(hashvalues)
    return float(k) / np.sum(hashvalues / float(MAX_HASH)) - 1.0


# ----------------------------------------------------------------------------
# LeanMinHash codec
# ----------------------------------------------------------------------------
def lean_bytesize(num_perm: int, byteorder: str = "@") -> int:
    """datasketch/lean_minhash.py:118-124: 'q' seed + 'i' count + K * 'I'."""
    return (struct.calcsize(byteorder + "q") + struct.calcsize(byteorder + "i")
            + num_perm * struct.calcsize(byteorder + "I"))


def lean_serialize(seed: int, hashvalues: np.ndarray, byteorder: str = "@") -> bytes:
    """datasketch/lean_minhash.py:174-175: struct '<bo>qi{K}I' of the hash values.

    ``struct`` 'I' refuses values >= 2^32, so (like the reference) this only works
    for signatures whose values fit 32 bits -- which MinHash guarantees.
    """
    k = len(hashvalues)
    buf = bytearray(struct.calcsize("%sqi%dI" % (byteorder, k)))
    struct.pack_into("%sqi%dI" % (byteorder, k), buf, 0, seed, k, *[int(x) for x in hashvalues])
    return bytes(buf)


def lean_deserialize(buf: bytes, byteorder: str = "@") -> Tuple[int, np.ndarray]:
    """datasketch/lean_minhash.py:201-214."""
    seed, k = struct.unpack_from("%sqi" % byteorder, buf, 0)
    off = struct.calcsize("%sqi" % byteorder)
    vals = struct.unpack_from(byteorder + "%dI" % k, buf, off)
    return seed, np.array(vals, dtype=np.uint64)


# ----------------------------------------------------------------------------
# Weighted MinHash (Ioffe ICWS)
# ----------------------------------------------------------------------------
def wmh_params(dim: int, sample_size: int, seed: int):
    """(rs, ln_cs, betas), each (sample_size, dim) float32.

    datasketch/weighted_minhash.py:118-121: one RandomState(seed); gamma(2,1),
    log(gamma(2,1)), uniform(0,1) drawn in that order, each cast to float32.
    """
    g = np.random.RandomState(seed=seed)
    rs = g.gamma(2, 1, (sample_size, dim)).astype(np.float32)
    ln_cs = np.log(g.gamma(2, 1, (sample_size, dim))).astype(np.float32)
    betas = g.uniform(0, 1, (sample_size, dim)).astype(np.float32)
    return rs, ln_cs, betas


def wmh_minhash(v, rs: np.ndarray, ln_cs: np.ndarray, betas: np.ndarray) -> np.ndarray:
    """(sample_size, 2) int64 of (k, t_k) (datasketch/weighted_minhash.py:136-158).

    Each float32 op is a separate rounding, in exactly this order:
    t = floor((vlog / r) + beta); ln_y = (t - beta) * r; ln_a = (ln_c - ln_y) - r;
    k = first index of the NaN-skipping minimum.
    """
    ss, dim = rs.shape
    if not hasattr(v, "__len__"):
        raise TypeError("Input vector must be sized")
    if len(v) != dim:
        raise ValueError("Input dimension mismatch, expecting %d" % dim)
    v = np.array(v, dtype=np.float32)  # always a private float32 copy
    out = np.zeros((ss, 2), dtype=int)
    z = v == 0
    if z.all():
        raise ValueError("Input is all zeros")
    v[z] = np.nan
    vlog = np.log(v)
    for i in range(ss):
        t = np.floor((vlog / rs[i]) + betas[i])
        ln_y = (t - betas[i]) * rs[i]
        ln_a = ln_cs[i] - ln_y - rs[i]
        k = np.nanargmin(ln_a)
        out[i][0], out[i][1] = k, int(t[k])
    return out


def wmh_minhash_many(X, rs: np.ndarray, ln_cs: np.ndarray, betas: np.ndarray) -> list:
    """Per row of X: (sample_size, 2) int array of (k, t_k), or None for an all-zero row
    (datasketch/weighted_minhash.py:161-247, the experimental batch method).

    Same sampling as ``wmh_minhash`` but the float32 roundings differ (:221-224):
    t = floor((log x / r) + beta); ln_y = ((t - beta) + 1) * r; ln_a = ln_c - ln_y; the argmin runs
    over the row's non-zero columns in index order (first minimum wins, :234-235).
    """
    X = np.asarray(X.toarray() if hasattr(X, "toarray") else X)
    if X.ndim != 2:
        raise ValueError("Input must have two dimensions")
    ss, dim = rs.shape
    if X.shape[1] != dim:
        raise ValueError("Input dimension mismatch, expecting %d" % dim)
    X = X.astype(np.float32)
    ret = []
    for row in X:
        cidx = np.nonzero(row)[0]
        if cidx.size == 0:
            ret.append(None)
            continue
        log_data = np.log(row[cidx])                    # float32
        r, be, lc = rs[:, cidx], betas[:, cidx], ln_cs[:, cidx]
        t = np.floor(log_data[None, :] / r + be)
        ln_y = (t - be + 1) * r
        ln_a = lc - ln_y
        am = np.argmin(ln_a, axis=1)
        out = np.zeros((ss, 2), dtype=int)
        out[:, 0] = cidx[am]
        out[:, 1] = t[np.arange(ss), am]
        ret.append(out)
    return ret


def wmh_jaccard(hv1: np.ndarray, hv2: np.ndarray) -> float:
    """Fraction of samples with equal (k,t) rows (datasketch/weighted_minhash.py:55-60)."""
    inter = 0
    for x, y in zip(hv1, hv2):
        if np.array_equal(x, y):
            inter += 1
    return float(inter) / float(len(hv1))


# ----------------------------------------------------------------------------
# MinHashLSH: parameters, band keys, dict bucketing
# ----------------------------------------------------------------------------
def _fp_prob(threshold: float, b: int, r: int) -> float:
    """datasketch/lsh.py:21-24."""
    from scipy.integrate import quad
    val, _ = quad(lambda s: 1 - (1 - s ** float(r)) ** float(b), 0.0, threshold)
    return val


def _fn_prob(threshold: float, b: int, r: int) -> float:
    """datasketch/lsh.py:27-30."""
    from scipy.integrate import quad
    val, _ = quad(lambda s: 1 - (1 - (1 - s ** float(r)) ** float(b)), threshold, 1.0)
    return val


def lsh_optimal_param(threshold: float, num_perm: int, fp_weight: float = 0.5,
                      fn_weight: float = 0.5) -> Tuple[int, int]:
    """(b, r) grid search (datasketch/lsh.py:33-48); first strict minimum wins."""
    best = float("inf")
    opt = (0, 0)
    for b in range(1, num_perm + 1):
        for r in range(1, int(num_perm / b) + 1):
            err = _fp_prob(threshold, b, r) * fp_weight + _fn_prob(threshold, b, r) * fn_weight
            if err < best:
                best = err
                opt = (b, r)
    return opt


def lsh_hashranges(b: int, r: int) -> List[Tuple[int, int]]:
    """datasketch/lsh.py:199."""
    return [(i * r, (i + 1) * r) for i in range(b)]


def lsh_band_key(band_values: np.ndarray) -> bytes:
    """Default ``_H`` = byteswap -> bytes (datasketch/lsh.py:537-538).

    For uint64 signatures this is the r values as big-endian 8-byte words.
    """
    return bytes(band_values.byteswap().data)


def lsh_band_keys(hashvalues: np.ndarray, b: int, r: int) -> List[bytes]:
    """All b keys of one signature (datasketch/lsh.py:344)."""
    return [lsh_band_key(hashvalues[s:e]) for s, e in lsh_hashranges(b, r)]


def bloom_band_keys(hashvalues: np.ndarray, b: int, r: int) -> np.ndarray:
    """The b Bloom keys of one signature: ``sum(hashvalues[start:end]) % _mersenne_prime`` per band
    (datasketch/lsh_bloom.py:105, :116; ``_mersenne_prime`` = 2**61 - 1, :20; hashranges :299)."""
    hv = np.asarray(hashvalues, dtype=np.uint64)
    p = (1 << 61) - 1
    return np.array([sum(int(x) for x in hv[s:e]) % p for s, e in lsh_hashranges(b, r)], dtype=np.uint64)


def redis_layout(keys, signatures: np.ndarray, b: int, r: int, basename: bytes, prepickle: bool = True) -> dict:
    """Database state of the reference's Redis-backed MinHashLSH after ``insert(key_i, signature_i)``:
    containers ``basename + b"_keys"`` / ``basename + b"_bucket_" + pack(">H", i)`` (datasketch/lsh.py:191-200),
    ``HSET name key -> name+key`` + ``RPUSH name+key H...`` (storage.py:1002-1004) for the keys container,
    ``HSET name_i H -> name_i+H`` + ``SADD name_i+H key`` (:1042-1045) per band; keys pickled when prepickle (lsh.py:340-341)."""
    import pickle
    import struct
    state = {"hash": {}, "list": {}, "set": {}}
    kname = basename + b"_keys"
    for key, hv in zip(keys, signatures):
        key = pickle.dumps(key) if prepickle else key
        hs = lsh_band_keys(np.asarray(hv, dtype=np.uint64), b, r)
        state["hash"].setdefault(kname, {})[key] = kname + key
        state["list"].setdefault(kname + key, []).extend(hs)
        for i, h in enumerate(hs):
            name = basename + b"_bucket_" + struct.pack(">H", i)
            state["hash"].setdefault(name, {})[h] = name + h
            state["set"].setdefault(name + h, set()).add(key)
    state["set"] = {k: sorted(v) for k, v in state["set"].items()}
    return state


class DictLSH:
    """Dict-storage MinHashLSH insert/query semantics.

    datasketch/lsh.py:326-347 (insert), :370-432 (query), over
    datasketch/storage.py:209-259 (defaultdict(list) keys, defaultdict(set) buckets).
    """

    def __init__(self, num_perm: int, b: int, r: int):
        from collections import defaultdict
        self.h, self.b, self.r = num_perm, b, r
        self.hashranges = lsh_hashranges(b, r)
        self.hashtables = [defaultdict(set) for _ in range(b)]
        self.keys = defaultdict(list)

    def insert(self, key, hashvalues: np.ndarray, check_duplication: bool = True):
        if len(hashvalues) != self.h:
            raise ValueError("Expecting minhash with length %d, got %d" % (self.h, len(hashvalues)))
        if check_duplication and key in self.keys:
            raise ValueError("The given key already exists")
        hs = [lsh_band_key(hashvalues[s:e]) for s, e in self.hashranges]
        self.keys[key].extend(hs)
        for h, table in zip(hs, self.hashtables):
            table[h].add(key)

    def query(self, hashvalues: np.ndarray) -> set:
        if len(hashvalues) != self.h:
            raise ValueError("Expecting minhash with length %d, got %d" % (self.h, len(hashvalues)))
        cand = set()
        for (s, e), table in zip(self.hashranges, self.hashtables):
            for key in table.get(lsh_band_key(hashvalues[s:e]), ()):
                cand.add(key)
        return cand


# ----------------------------------------------------------------------------
# hashfunc (host-side by the reference's contract; restated for fixtures)
# ----------------------------------------------------------------------------
def sha1_hash32(data: bytes) -> int:
    """First 4 bytes of SHA1, little-endian (datasketch/hashfunc.py:15)."""
    import hashlib
    return struct.unpack("<I", hashlib.sha1(data).digest()[:4])[0]


# ----------------------------------------------------------------------------
# Scalar big-int cross-check used by the adversarial tests
# ----------------------------------------------------------------------------
def permute_scalar(a: int, b: int, h: int) -> int:
    """Python big-int statement of numpy's uint64 semantics for one evaluation:
    ((a*h + b) mod 2^64) mod (2^61-1), low 32 bits (minhash.py:223 / :295-296)."""
    x = (a * h + b) & ((1 << 64) - 1)
    return (x % ((1 << 61) - 1)) & 0xFFFFFFFF


# ----------------------------------------------------------------------------
# Non-cryptographic token hashes the reference documents as `hashfunc` choices
# (docs/minhash.rst:79-112).  Third-party algorithms, absent from the reference's
# tree: xxHash 32-bit (package `xxhash`, pinned by tests/golden/hashes.npz which
# that package produced) and MurmurHash3 x86_32 (package `mmh3`, not installed
# here: pinned by its published verification vectors in tests/test_oracle_golden.py).
# Restated with numpy uint32 scalars (wrap-around arithmetic).
# ----------------------------------------------------------------------------
def _u32(x):
    return np.uint32(int(x) & 0xFFFFFFFF)


def _rol(x, n):
    x = int(x)
    return _u32((x << n) | (x >> (32 - n)))


def xxh32(data: bytes, seed: int = 0) -> int:
    d = np.frombuffer(bytes(data), dtype=np.uint8)
    n = len(d)
    P1, P2, P3, P4, P5 = (_u32(v) for v in (2654435761, 2246822519, 3266489917, 668265263, 374761393))
    words = d[: n // 4 * 4].view("<u4") if n >= 4 else np.zeros(0, dtype=np.uint32)
    with np.errstate(over="ignore"):
        s32 = _u32(seed)
        w = 0
        if n >= 16:
            acc = [s32 + P1 + P2, s32 + P2, s32, s32 - P1]
            for stripe in range(n // 16):
                for lane in range(4):
                    acc[lane] = _rol(acc[lane] + words[4 * stripe + lane] * P2, 13) * P1
            w = 4 * (n // 16)
            h = _rol(acc[0], 1) + _rol(acc[1], 7) + _rol(acc[2], 12) + _rol(acc[3], 18)
        else:
            h = s32 + P5
        h = h + _u32(n)
        for q in range(w, n // 4):
            h = _rol(h + words[q] * P3, 17) * P4
        for byte in d[n // 4 * 4:]:
            h = _rol(h + _u32(byte) * P5, 11) * P1
        h = (h ^ (h >> np.uint32(15))) * P2
        h = (h ^ (h >> np.uint32(13))) * P3
        h = h ^ (h >> np.uint32(16))
    return int(h)


def murmur3_32(data: bytes, seed: int = 0) -> int:
    d = np.frombuffer(bytes(data), dtype=np.uint8)
    n = len(d)
    C1, C2 = _u32(0xCC9E2D51), _u32(0x1B873593)
    with np.errstate(over="ignore"):
        h = _u32(seed)
        for k in (d[: n // 4 * 4].view("<u4") if n >= 4 else []):
            k = _rol(k * C1, 15) * C2
            h = _rol(h ^ k, 13) * np.uint32(5) + _u32(0xE6546B64)
        tail = d[n // 4 * 4:]
        if len(tail):
            k = _u32(sum(int(b) << (8 * i) for i, b in enumerate(tail)))
            h = h ^ (_rol(k * C1, 15) * C2)
        h = h ^ _u32(n)
        h = (h ^ (h >> np.uint32(16))) * _u32(0x85EBCA6B)
        h = (h ^ (h >> np.uint32(13))) * _u32(0xC2B2AE35)
        h = h ^ (h >> np.uint32(16))
    return int(h)
