"""TEST INFRASTRUCTURE ONLY -- API-behaviour scenarios run on a `datasketch`-like module.

Each scenario drives the public API (MinHash, LeanMinHash, MinHashLSH, MinHashLSHForest) through ordinary use and
through misuse, and returns what a caller observes as plain JSON values: numbers, sorted key lists, byte strings as hex,
and the exception type a call raises.  oracle/gen_api_golden.py runs them on the reference and stores the result in
tests/golden/api_behaviour.json; tests/test_api_behaviour.py runs them on datasketch_b200 and compares.
"""
from __future__ import annotations

import hashlib
import pickle

import numpy as np


def enc(x):
    if isinstance(x, np.ndarray):
        return [int(v) for v in x.reshape(-1)]
    if isinstance(x, (bytes, bytearray, memoryview)):
        return bytes(x).hex()
    if isinstance(x, (set, frozenset)):
        return sorted(enc(v) for v in x)
    if isinstance(x, (list, tuple)):
        return [enc(v) for v in x]
    if isinstance(x, dict):
        return {str(k): enc(v) for k, v in sorted(x.items(), key=lambda kv: str(kv[0]))}
    if isinstance(x, (bool, np.bool_)):
        return bool(x)
    if isinstance(x, (int, np.integer)):
        return int(x)
    if isinstance(x, (float, np.floating)):
        return float(x)
    return x


def call(fn):
    """What the caller sees: the encoded result, or {"raises": <exception type name>}."""
    try:
        return enc(fn())
    except Exception as exc:  # noqa: BLE001
        return {"raises": type(exc).__name__}


def _words(n, seed):
    rs = np.random.RandomState(seed)
    return [("w%d" % v).encode() for v in rs.randint(0, 4 * n, size=n)]


def _mh(ds, words, num_perm=128, seed=1):
    m = ds.MinHash(num_perm=num_perm, seed=seed)
    m.update_batch(words)
    return m


def minhash_basics(ds):
    a, b = _words(300, 1), _words(300, 2)
    m1, m2 = _mh(ds, a), _mh(ds, a[:150] + b[:150])
    e = ds.MinHash(num_perm=128, seed=1)
    r = {"empty": call(e.is_empty), "len": call(lambda: len(m1)), "digest": call(m1.digest),
         "jaccard": call(lambda: m1.jaccard(m2)), "count": call(m1.count), "not_empty": call(m1.is_empty),
         "eq_self_copy": call(lambda: m1 == m1.copy()), "eq_other": call(lambda: m1 == m2)}
    m3 = ds.MinHash(num_perm=128, seed=1)
    for w in a:
        m3.update(w)
    r["update_equals_batch"] = call(lambda: m3 == m1)
    mm = m1.copy()
    mm.merge(m2)
    r["merge"] = call(mm.digest)
    r["union"] = call(lambda: ds.MinHash.union(m1, m2).digest())
    r["union_eq_merge"] = call(lambda: ds.MinHash.union(m1, m2) == mm)
    c = m1.copy()
    c.clear()
    r["clear"] = call(lambda: (c.is_empty(), c.digest()))
    r["jaccard_empty"] = call(lambda: e.jaccard(ds.MinHash(num_perm=128, seed=1)))
    r["count_empty"] = call(e.count)
    return r


def minhash_misuse(ds):
    m = _mh(ds, _words(50, 3))
    r = {"jaccard_other_seed": call(lambda: m.jaccard(_mh(ds, _words(50, 3), seed=2))),
         "jaccard_other_num_perm": call(lambda: m.jaccard(_mh(ds, _words(50, 3), num_perm=64))),
         "merge_other_seed": call(lambda: m.copy().merge(_mh(ds, _words(50, 3), seed=2))),
         "merge_other_num_perm": call(lambda: m.copy().merge(_mh(ds, _words(50, 3), num_perm=64))),
         "union_one": call(lambda: ds.MinHash.union(m).digest()),
         "union_other_seed": call(lambda: ds.MinHash.union(m, _mh(ds, _words(5, 4), seed=2))),
         "num_perm_too_large": call(lambda: ds.MinHash(num_perm=2 ** 32 + 1)),
         "hashvalues_and_permutations_mismatch": call(
             lambda: ds.MinHash(num_perm=4, hashvalues=np.ones(5, dtype=np.uint64)).digest()),
         "from_hashvalues": call(lambda: ds.MinHash(hashvalues=m.hashvalues).digest()),
         "from_hashvalues_eq": call(lambda: ds.MinHash(hashvalues=m.hashvalues, seed=1) == m)}
    return r


def sha1_low32(b):
    """A caller's own hash function (module level, so MinHash objects that use it pickle)."""
    return int.from_bytes(hashlib.sha1(b).digest()[:4], "little")


def minhash_bulk_and_pickle(ds):
    docs = [_words(n, 10 + n) for n in (0, 1, 7, 200)]
    bulk = ds.MinHash.bulk(docs, num_perm=64, seed=5, hashfunc=sha1_low32)
    gen = list(ds.MinHash.generator(docs, num_perm=64, seed=5, hashfunc=sha1_low32))
    one = []
    for d in docs:
        m = ds.MinHash(num_perm=64, seed=5, hashfunc=sha1_low32)
        m.update_batch(d)
        one.append(m)
    m = _mh(ds, _words(100, 9))
    p = pickle.loads(pickle.dumps(m))
    return {"bulk": call(lambda: [x.digest() for x in bulk]),
            "bulk_eq_single": call(lambda: [x == y for x, y in zip(bulk, one)]),
            "generator_eq_bulk": call(lambda: [x == y for x, y in zip(gen, bulk)]),
            "pickle_eq": call(lambda: p == m), "pickle_seed": call(lambda: p.seed),
            "pickle_digest": call(p.digest)}


def lean_minhash(ds):
    m = _mh(ds, _words(120, 11), num_perm=64, seed=3)
    lm = ds.LeanMinHash(m)
    r = {"seed": call(lambda: lm.seed), "digest": call(lm.digest), "eq_minhash": call(lambda: lm == m),
         "jaccard": call(lambda: lm.jaccard(ds.LeanMinHash(_mh(ds, _words(120, 12), num_perm=64, seed=3)))),
         "count": call(lm.count), "bytesize": call(lm.bytesize), "bytesize_le": call(lambda: lm.bytesize("<")),
         "update": call(lambda: lm.update(b"x"))}
    for bo in ("<", ">", "!"):
        buf = bytearray(lm.bytesize(bo))
        lm.serialize(buf, bo)
        r["serialize" + bo] = enc(buf)
        r["roundtrip" + bo] = call(lambda: ds.LeanMinHash.deserialize(buf, bo) == lm)
    r["serialize_short_buffer"] = call(lambda: lm.serialize(bytearray(8)))
    r["pickle_eq"] = call(lambda: pickle.loads(pickle.dumps(lm)) == lm)
    r["union"] = call(lambda: ds.LeanMinHash.union(lm, ds.LeanMinHash(_mh(ds, _words(9, 13), num_perm=64, seed=3)))
                      .digest())
    r["from_seed_hashvalues"] = call(lambda: ds.LeanMinHash(seed=3, hashvalues=m.hashvalues) == lm)
    r["empty_constructor"] = call(lambda: ds.LeanMinHash())
    return r


def _lsh_data(ds, num_perm=128):
    base = _words(200, 20)
    docs = {"k%d" % i: base[: 200 - 12 * i] + _words(12 * i, 30 + i) for i in range(12)}
    return {k: _mh(ds, v, num_perm=num_perm) for k, v in docs.items()}


def lsh(ds):
    ms = _lsh_data(ds)
    lsh_ = ds.MinHashLSH(threshold=0.6, num_perm=128)
    r = {"params": call(lambda: [lsh_.b, lsh_.r]), "empty": call(lsh_.is_empty)}
    for k, m in ms.items():
        lsh_.insert(k, m)
    q = ms["k3"]
    r["query"] = call(lambda: sorted(lsh_.query(q)))
    r["contains"] = call(lambda: ["k3" in lsh_, "nope" in lsh_])
    r["insert_duplicate_key"] = call(lambda: lsh_.insert("k3", q))
    r["insert_other_num_perm"] = call(lambda: lsh_.insert("z", _mh(ds, _words(10, 1), num_perm=64)))
    r["query_other_num_perm"] = call(lambda: lsh_.query(_mh(ds, _words(10, 1), num_perm=64)))
    r["counts"] = call(lambda: [sorted(d.values()) for d in lsh_.get_counts()])
    r["subset_counts"] = call(lambda: [sorted(d.values()) for d in lsh_.get_subset_counts("k0", "k1")])
    lsh_.remove("k3")
    r["after_remove"] = call(lambda: (sorted(lsh_.query(q)), "k3" in lsh_))
    r["remove_missing"] = call(lambda: lsh_.remove("k3"))
    r["pickle_query"] = call(lambda: sorted(pickle.loads(pickle.dumps(lsh_)).query(ms["k0"])))
    s = ds.MinHashLSH(threshold=0.6, num_perm=128)
    with s.insertion_session() as sess:
        for k, m in ms.items():
            sess.insert(k, m)
    r["session_query"] = call(lambda: sorted(s.query(ms["k5"])))
    r["weights_params"] = call(lambda: [ds.MinHashLSH(threshold=0.5, num_perm=128, weights=(0.2, 0.8)).b,
                                        ds.MinHashLSH(threshold=0.5, num_perm=128, weights=(0.2, 0.8)).r])
    r["explicit_params"] = call(lambda: [ds.MinHashLSH(num_perm=128, params=(16, 8)).b,
                                         ds.MinHashLSH(num_perm=128, params=(16, 8)).r])
    r["bad_threshold"] = call(lambda: ds.MinHashLSH(threshold=1.5, num_perm=128))
    r["bad_params"] = call(lambda: ds.MinHashLSH(num_perm=128, params=(20, 8)))
    r["bad_weights"] = call(lambda: ds.MinHashLSH(threshold=0.5, num_perm=128, weights=(0.2, 0.2)))
    m = ds.MinHashLSH(threshold=0.6, num_perm=128)
    m.insert("k0", ms["k0"])
    other = ds.MinHashLSH(threshold=0.6, num_perm=128)
    other.insert("k1", ms["k1"])
    m.merge(other)
    r["merge_query"] = call(lambda: sorted(m.query(ms["k0"])))
    r["merge_overlap"] = call(lambda: m.merge(other, check_overlap=True))
    return r


def lsh_forest(ds):
    ms = _lsh_data(ds)
    f = ds.MinHashLSHForest(num_perm=128, l=8)
    r = {"empty": call(f.is_empty)}
    for k, m in ms.items():
        f.add(k, m)
    r["query_before_index"] = call(lambda: sorted(f.query(ms["k0"], 3)))
    f.index()
    r["top3"] = call(lambda: sorted(f.query(ms["k0"], 3)))
    r["top1"] = call(lambda: f.query(ms["k11"], 1))
    r["top_all"] = call(lambda: sorted(f.query(ms["k4"], 50)))
    r["k_zero"] = call(lambda: f.query(ms["k4"], 0))
    r["contains"] = call(lambda: ["k4" in f, "nope" in f])
    r["add_duplicate"] = call(lambda: f.add("k4", ms["k4"]))
    r["add_other_num_perm"] = call(lambda: f.add("z", _mh(ds, _words(10, 1), num_perm=64)))
    r["hashvalues"] = call(lambda: f.get_minhash_hashvalues("k2"))
    r["pickle_top3"] = call(lambda: sorted(pickle.loads(pickle.dumps(f)).query(ms["k0"], 3)))
    return r


SCENARIOS = {f.__name__: f for f in (minhash_basics, minhash_misuse, minhash_bulk_and_pickle, lean_minhash, lsh,
                                      lsh_forest)}
