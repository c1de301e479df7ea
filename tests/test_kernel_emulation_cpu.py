"""The CUDA signature kernel's own source, run on the CPU against the oracle.

``tests/emu/`` compiles ``datasketch_b200/csrc/signature_kernel.cu``, ``minhash_kernels.cu`` and ``codec_kernels.cu`` -- kernels AND launchers --
with g++ (``-DDSK_EMU``): every CUDA thread is a host thread, warp / CTA barriers are pthread barriers, and the async
bulk copies are emulated adversarially (destination poisoned at issue, data delivered only when a waiter polls the
mbarrier, shared->global stores deferred until ``bulk_wait_read``).  What this checks is the *logic* -- the per-warp
ring protocol, block patching at document boundaries, the array's <16-byte tail, dynamic work units, the two-phase
tracking, the warp-wide exact path for flagged permutations and the de-duplicating stage, init merging, K slicing, the launchers' choices, the 4-stage TMA tile pipeline of
the LeanMinHash codec -- on the exact source that nvcc compiles for the B200 (the hooks are preprocessor-only; the
product's SASS is byte-identical with and without them).  It says nothing about performance, and the GPU tests remain
the parity gate for the compiled kernels.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import oracle_clib as oc
from oracle import oracle_np as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu")
TWO_PHASE, DIRECT, EXACT = 0, 1, 2

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")


@pytest.fixture(scope="module")
def emu():
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemu_kernels.so")
    srcs = [os.path.join(EMU, "emu_kernels.cpp"), os.path.join(EMU, "cuda_emu.h"),
            os.path.join(ROOT, "datasketch_b200", "csrc", "minhash_kernels.cu"),
            os.path.join(ROOT, "datasketch_b200", "csrc", "signature_kernel.cu"),
            os.path.join(ROOT, "datasketch_b200", "csrc", "dsk_common.cuh")] + [
                os.path.join(ROOT, "datasketch_b200", "csrc", f + "_kernels.cu") for f in ("codec", "lsh", "jaccard", "sha1", "hash", "wmh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-std=c++17", "-O1", "-pthread", "-ffp-contract=off", "-DDSK_EMU", "-I" + EMU, "-shared", "-fPIC", "-o", so,
                        srcs[0]], check=True)
    lib = ctypes.CDLL(so)
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.emu_minhash_bulk.argtypes = [vp, ci, vp, i64, vp, vp, ci, ci, ci, vp, i64, ci, vp, ci, ci, ci, ci]
    lib.emu_minhash_bulk.restype = ci

    def run(tok, off, perms, mode, v1=0, init=None, out_u64=False, docs_per_unit=3, grid_x=1, gen=0):
        k, n = perms.shape[1], len(off) - 1
        tok = np.ascontiguousarray(tok)
        off = np.ascontiguousarray(off, dtype=np.int64)
        out = np.zeros((n, k), dtype=np.uint64 if out_u64 else np.uint32)
        a, b = np.ascontiguousarray(perms[0]), np.ascontiguousarray(perms[1])
        ip, stride, i64f = None, 0, 0
        if init is not None:
            init = np.ascontiguousarray(init)
            ip, stride, i64f = init.ctypes.data, (0 if init.ndim == 1 else k), int(init.dtype == np.uint64)
        rc = lib.emu_minhash_bulk(tok.ctypes.data, int(tok.dtype == np.uint64), off.ctypes.data, n, a.ctypes.data,
                                  b.ctypes.data, k, mode, v1, ip, stride, i64f, out.ctypes.data, int(out_u64),
                                  docs_per_unit, grid_x, gen)
        assert rc == 0
        return out
    def stats():
        buf = (ctypes.c_longlong * 5)()
        lib.emu_sig_stats(buf)
        return dict(zip(("in_place", "copied", "deduped", "removed", "flagged"), list(buf)))
    run.lib = lib
    run.stats = stats
    return run


def _ragged(rs, n, maxlen, extra_tail=0):
    lens = rs.randint(0, maxlen + 1, size=n)
    lens[:5] = [0, 1, 15, 16, 17]
    lens[-1] = 0
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    off[-1] += extra_tail                      # makes the token count not a multiple of 4 (the <16-byte array tail)
    tok = rs.randint(0, 1 << 32, size=int(off[-1]), dtype=np.uint64).astype(np.uint32)
    return tok, off


@pytest.mark.parametrize("k", [16, 64, 100, 128, 192, 256, 300])
def test_all_modes_ragged_documents(emu, k):
    rs = np.random.RandomState(k)
    tok, off = _ragged(rs, 60, 150, extra_tail=3)
    perms = o.init_permutations(k, 1)
    want = oc.minhash_bulk_u32tok(tok, off, perms)
    for mode in (TWO_PHASE, DIRECT, EXACT):
        assert np.array_equal(emu(tok, off, perms, mode), want), (k, mode)
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE, v1=1), want)


@pytest.mark.parametrize("v1", [0, 1])
@pytest.mark.parametrize("share", [0.05, 0.6])
def test_repeated_tokens_stay_exact(emu, v1, share):
    rs = np.random.RandomState(int(share * 100) + v1)
    tok, off = _ragged(rs, 50, 400, extra_tail=1)
    for d in range(len(off) - 1):
        a, b = int(off[d]), int(off[d + 1])
        if b - a > 1:
            rep = np.nonzero(rs.uniform(size=b - a) < share)[0]
            rep = rep[rep > 0]
            tok[a + rep] = tok[a + (rs.uniform(size=len(rep)) * rep).astype(np.int64)]
    for k in (128, 256):
        perms = o.init_permutations(k, 2)
        assert np.array_equal(emu(tok, off, perms, TWO_PHASE, v1=v1), oc.minhash_bulk_u32tok(tok, off, perms))


@pytest.mark.parametrize("v1", [0, 1])
def test_structured_tokens_small_minimum_and_wrap(emu, v1):
    """Tiny and near-2^32 tokens: products next to the wrap, min L' < 7 cases, many exact ties."""
    tok = np.concatenate([np.arange(0, 3000, dtype=np.uint32),
                          (np.uint64(1 << 32) - np.arange(1, 3001, dtype=np.uint64)).astype(np.uint32),
                          np.zeros(500, dtype=np.uint32), np.full(500, 0xFFFFFFFF, dtype=np.uint32)])
    off = np.arange(0, len(tok) + 1, 125, dtype=np.int64)
    perms = o.init_permutations(128, 3)
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE, v1=v1), oc.minhash_bulk_u32tok(tok, off, perms))


def test_long_documents_leave_the_ring_and_units_of_every_size(emu):
    """Documents far longer than the 3 x 2 KB ring (winners evicted before phase 2), unit sizes 1 / 5 / 32, two CTAs."""
    rs = np.random.RandomState(8)
    lens = np.array([5000, 3, 2049, 0, 1537, 4096, 7, 2600], dtype=np.int64)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rs.randint(0, 1 << 32, size=int(off[-1]), dtype=np.uint64).astype(np.uint32)
    perms = o.init_permutations(128, 1)
    want = oc.minhash_bulk_u32tok(tok, off, perms)
    for dpu, gx in ((1, 2), (5, 1), (32, 2)):
        for v1 in (0, 1):
            assert np.array_equal(emu(tok, off, perms, TWO_PHASE, v1=v1, docs_per_unit=dpu, grid_x=gx), want)
    assert np.array_equal(emu(tok, off, perms, DIRECT, docs_per_unit=2, grid_x=2), want)


@pytest.mark.parametrize("T", [16, 64, 256, 512, 528, 1040])
def test_aligned_documents_use_the_ring_in_place(emu, T):
    """Documents whose length is a multiple of 16 and whose start is 16-byte aligned are read straight from the ring
    (signature_kernel.cu "in place"); the ones that would wrap the 1024-token ring, and every sub-piece after an odd
    one, take the copy.  A 4-token shift of the whole batch changes which documents wrap."""
    rs = np.random.RandomState(T)
    n = 37
    for lead in (0, 4, 20):                     # one leading document of `lead` tokens shifts everything behind it
        lens = np.full(n, T, dtype=np.int64)
        lens[0] = lead
        off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lens, out=off[1:])
        tok = rs.randint(0, 1 << 32, size=int(off[-1]), dtype=np.uint64).astype(np.uint32)
        for k in (128, 256):
            perms = o.init_permutations(k, 1)
            want = oc.minhash_bulk_u32tok(tok, off, perms)
            for dpu, gx in ((32, 1), (5, 2)):
                emu.stats()
                assert np.array_equal(emu(tok, off, perms, TWO_PHASE, docs_per_unit=dpu, grid_x=gx), want), (T, lead, k, dpu)
                st = emu.stats()
                assert st["in_place"] > 0 and st["deduped"] == 0, st
                if lead == 0 and T in (16, 64, 256, 512):      # nothing wraps, nothing is ragged: never copied
                    assert st["copied"] == 0, st
                if T == 1040 or lead == 20:
                    assert st["copied"] > 0, st


def test_deduplication_switches_on_and_off(emu):
    """Repeated tokens tie across blocks; after a sub-piece with >= 4 flagged permutations the warp deduplicates while
    it stages, and stops again after 16 sub-pieces in which nothing was removed.  One warp (grid 1 x 1 CTA, one
    unit) walks: clean -> heavy repeats -> clean (long enough to switch off) -> repeats again; 0xFFFFFFFF tokens
    (the hash set's empty marker) are repeated too."""
    rs = np.random.RandomState(77)
    lens = [256] * 4 + [300] * 6 + [256] * 40 + [190] * 4 + [1200, 256]
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rs.randint(0, 1 << 32, size=int(off[-1]), dtype=np.uint64).astype(np.uint32)
    for d in list(range(4, 10)) + list(range(50, 55)):
        a, b = int(off[d]), int(off[d + 1])
        pool = tok[a:a + max(8, (b - a) // 3)].copy()
        pool[0] = 0xFFFFFFFF
        tok[a:b] = pool[rs.randint(0, len(pool), size=b - a)]
    perms = o.init_permutations(128, 9)
    want = oc.minhash_bulk_u32tok(tok, off, perms)
    emu.stats()
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE, docs_per_unit=64, grid_x=1), want)
    st = emu.stats()
    # one warp walked everything: it staged in place first, flagged the repeats, de-duplicated (removing tokens),
    # went back to in-place staging during the 40 clean documents and de-duplicated again at the end
    assert st["flagged"] >= 8 and st["removed"] > 500 and 16 <= st["deduped"] < 45 and st["in_place"] >= 20, st
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE, docs_per_unit=7, grid_x=2), want)


@pytest.mark.parametrize("k", [128, 300])
def test_long_documents_are_cut_into_pieces_on_the_device(emu, k):
    """signature_kernel.cu piece mode (thresholds shrunk to 100 / 32 tokens so the emulation stays small): the warp that
    meets a long document stores the row's initial value and appends pieces; the second launch min-merges them with
    atomicMin.  Mixed with short / empty documents, running-state merge, u64 output, K sliced over blockIdx.y (k = 300)."""
    lib = emu.lib
    rs = np.random.RandomState(k)
    lens = np.array([30, 250, 0, 101, 100, 1000, 7, 99, 481, 40, 3000, 12], dtype=np.int64)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rs.randint(0, 1 << 32, size=int(off[-1]) + 3, dtype=np.uint64).astype(np.uint32)[:int(off[-1])]
    tok[off[5]:off[5] + 500] = tok[off[5] + 500:off[5] + 1000]          # repeats inside a long document
    perms = o.init_permutations(k, 4)
    a, b = np.ascontiguousarray(perms[0]), np.ascontiguousarray(perms[1])
    want = oc.minhash_bulk_u32tok(tok, off, perms)
    n = len(lens)
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.emu_minhash_sig_long.argtypes = [vp, vp, i64, vp, vp, ci, vp, i64, ci, vp, ci, ci, ci, i64, ci, vp, ci]
    npieces = ctypes.c_longlong(0)
    for dpu, gx in ((3, 1), (1, 2), (32, 2)):
        out = np.zeros((n, k), dtype=np.uint32)
        assert lib.emu_minhash_sig_long(tok.ctypes.data, off.ctypes.data, n, a.ctypes.data, b.ctypes.data, k, None, 0, 0,
                                        out.ctypes.data, 0, dpu, gx, 100, 5, ctypes.byref(npieces), 0) == 0
        assert np.array_equal(out, want), (dpu, gx)
        assert npieces.value == sum(-(-int(x) // 32) for x in lens if x > 100)      # 250, 101, 1000, 481, 3000
    init = rs.randint(0, 1 << 32, size=(n, k), dtype=np.uint64)
    out64 = np.zeros((n, k), dtype=np.uint64)
    assert lib.emu_minhash_sig_long(tok.ctypes.data, off.ctypes.data, n, a.ctypes.data, b.ctypes.data, k, init.ctypes.data, k, 1,
                                    out64.ctypes.data, 1, 2, 2, 100, 5, None, 0) == 0
    assert np.array_equal(out64, np.minimum(want.astype(np.uint64), init))


def test_u64_tokens_init_merge_and_u64_output(emu):
    rs = np.random.RandomState(4)
    tok32, off = _ragged(rs, 30, 90)
    k = 64
    perms = o.init_permutations(k, 5)
    tok64 = rs.randint(0, 1 << 63, size=len(tok32), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    want64 = oc.minhash_bulk_u64tok(tok64, off, perms)
    assert np.array_equal(emu(tok64, off, perms, EXACT), want64)
    base = oc.minhash_bulk_u32tok(tok32, off, perms)
    row = rs.randint(0, 1 << 32, size=k, dtype=np.uint64)
    mat = rs.randint(0, 1 << 32, size=base.shape, dtype=np.uint64)
    got = emu(tok32, off, perms, TWO_PHASE, init=row, out_u64=True)
    assert got.dtype == np.uint64 and np.array_equal(got, np.minimum(base.astype(np.uint64), row[None, :]))
    got = emu(tok32, off, perms, DIRECT, init=mat.astype(np.uint32))
    assert np.array_equal(got, np.minimum(base, mat.astype(np.uint32)))
    got = emu(tok32, off, perms, EXACT, init=mat, out_u64=True)
    assert np.array_equal(got, np.minimum(base.astype(np.uint64), mat))


def test_thread_sanitizer_finds_no_race_in_the_ring_protocol():
    """The emulated kernel under ThreadSanitizer (tests/emu/emu_tsan_main.cpp): a shared-memory access the kernel does not
    order with __syncwarp / the mbarrier -- a ring slot refilled while a lane still reads it, the scratch line reused
    too early -- shows up as a data race between the host threads that play the lanes.  (Control experiment, not
    committed: deleting the __syncwarp after the scratch-line write makes TSan report the race and the results differ.)"""
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    exe = os.path.join(out, "emu_tsan")
    build = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-pthread", "-ffp-contract=off", "-fsanitize=thread", "-DDSK_EMU", "-I" + EMU,
                            "-o", exe, os.path.join(EMU, "emu_kernels.cpp"), os.path.join(EMU, "emu_tsan_main.cpp")],
                           capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("ThreadSanitizer runtime not available: " + build.stderr[-200:])
    env = dict(os.environ, TSAN_OPTIONS="history_size=7 halt_on_error=1 exitcode=66")   # history: see emu_tsan_main.cpp
    run = subprocess.run([exe], capture_output=True, text=True, env=env, timeout=900)
    text = run.stdout + run.stderr
    if run.returncode not in (0, 1, 66) or "unexpected memory mapping" in text:
        pytest.skip("ThreadSanitizer cannot run in this container: " + text[-200:])
    assert "data race" not in text and run.returncode == 0, text[-2000:]
    assert text.count("identical") == 8


# ---- codec kernels (codec_kernels.cu): TMA tile pipeline and the simple kernels ----------------------------------
def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


@pytest.mark.parametrize("k,n", [(128, 1000), (4, 333), (100, 75), (256, 41), (10, 50)])
@pytest.mark.parametrize("bo", ["<", ">"])
def test_lean_codec_tile_pipeline_and_fallbacks(emu, k, n, bo):
    """k % 4 == 0 takes the 4-stage bulk-copy tile kernel (several tiles per CTA with sm_count = 1, ragged last tile),
    other k the per-word kernels; both byte orders; u64 input; header validation on unpack."""
    lib = emu.lib
    rs = np.random.RandomState(k + n)
    sig = rs.randint(0, 1 << 32, size=(n, k), dtype=np.uint64).astype(np.uint32)
    seed = -123456789012345 if k % 8 else 7
    big = int(bo == ">")
    rec = np.zeros((n, 12 + 4 * k), dtype=np.uint8)
    for sm_count in (1, 3):
        rec[:] = 0
        assert lib.emu_lean_pack(_ptr(sig), 0, n, k, ctypes.c_int64(seed), big, _ptr(rec), sm_count) == 0
        for i in (0, n // 2, n - 1):
            assert rec[i].tobytes() == o.lean_serialize(seed, sig[i].astype(np.uint64), bo)
        back = np.zeros_like(sig)
        status = np.zeros(1, dtype=np.int32)
        assert lib.emu_lean_unpack(_ptr(rec), n, k, ctypes.c_int64(seed), big, _ptr(back), 0, _ptr(status), sm_count) == 0
        assert status[0] == 0 and np.array_equal(back, sig)
    rec64 = np.zeros_like(rec)
    sig64 = sig.astype(np.uint64)
    assert lib.emu_lean_pack(_ptr(sig64), 1, n, k, ctypes.c_int64(seed), big, _ptr(rec64), 2) == 0
    assert np.array_equal(rec64, rec)
    back64 = np.zeros((n, k), dtype=np.uint64)
    status = np.zeros(1, dtype=np.int32)
    assert lib.emu_lean_unpack(_ptr(rec), n, k, ctypes.c_int64(seed + 1), big, _ptr(back64), 1, _ptr(status), 2) == 0
    assert status[0] == 1                                   # wrong seed in the header is flagged
    if bo == "<":
        assert np.array_equal(rec, oc.lean_pack_le(sig, seed))


@pytest.mark.parametrize("k,b,r", [(128, 9, 13), (128, 32, 4), (256, 17, 15), (16, 4, 4), (32, 32, 1)])
def test_band_keys_fingerprints_and_bbit_blocks(emu, golden, k, b, r):
    lib = emu.lib
    rs = np.random.RandomState(b * r)
    n = 97
    sig = rs.randint(0, 1 << 32, size=(n, k), dtype=np.uint64).astype(np.uint32)
    sig[1] = sig[0]
    keys = np.zeros((n, b, 8 * r), dtype=np.uint8)
    assert lib.emu_band_keys(_ptr(sig), n, k, b, r, _ptr(keys)) == 0
    assert np.array_equal(keys, oc.band_keys_be(sig, b, r))
    fp = np.zeros((n, b), dtype=np.uint64)
    assert lib.emu_band_fingerprints(_ptr(sig), n, k, b, r, _ptr(fp)) == 0
    assert np.array_equal(fp[0], fp[1]) and len(np.unique(fp)) >= (n - 1) * b - 2
    # b-bit blocks against the reference's pickle layout (tests/golden/bbit.npz pins the host class)
    import struct
    for bits, slot in ((1, 1), (2, 2), (3, 4), (8, 8), (13, 16), (32, 32)):
        per = 64 // slot
        nblk = -(-k // per)
        blocks = np.zeros((n, nblk), dtype=np.uint64)
        assert lib.emu_bbit_pack(_ptr(sig), n, k, bits, slot, _ptr(blocks)) == 0
        masked = sig & np.uint32((1 << bits) - 1) if bits < 32 else sig
        want0 = 0
        for j, v in enumerate(masked[0][:per]):
            want0 |= int(v) << (per - 1 - j) * slot
        assert int(blocks[0, 0]) == want0
        back = np.zeros_like(sig)
        assert lib.emu_bbit_unpack(_ptr(blocks), n, k, slot, _ptr(back)) == 0
        assert np.array_equal(back, masked)


def test_seg_min_and_merge_kernels(emu):
    lib = emu.lib
    rs = np.random.RandomState(2)
    k = 100
    seg = np.array([0, 3, 3, 4, 10], dtype=np.int64)        # document 1 has no piece
    part = rs.randint(0, 1 << 32, size=(10, k), dtype=np.uint64).astype(np.uint32)
    init = rs.randint(0, 1 << 32, size=(4, k), dtype=np.uint64)
    out = np.zeros((4, k), dtype=np.uint64)
    assert lib.emu_seg_min(_ptr(part), _ptr(seg), 4, k, _ptr(init), k, 1, _ptr(out), 1) == 0
    for d in range(4):
        rows = part[seg[d]:seg[d + 1]].astype(np.uint64)
        want = np.minimum(init[d], rows.min(axis=0)) if len(rows) else np.minimum(init[d], np.uint64(0xFFFFFFFF))
        assert np.array_equal(out[d], want)
    x = rs.randint(0, 1 << 32, size=5000, dtype=np.uint64).astype(np.uint32)
    y = rs.randint(0, 1 << 32, size=5000, dtype=np.uint64).astype(np.uint32)
    z = np.zeros_like(x)
    assert lib.emu_sig_merge_min(_ptr(x), _ptr(y), 5000, _ptr(z)) == 0 and np.array_equal(z, np.minimum(x, y))


# ---- LSH index, forest, Jaccard, SHA1, Weighted MinHash kernels -------------------------------------------------------
def test_lsh_insert_query_kernels_vs_dict_oracle(emu):
    """dsk_lsh_*'s kernels (atomicCAS-claimed open-addressing tables, atomicExch bucket chains, tuple verification,
    count -> scan -> fill) against the reference's dict buckets: candidate sets must be identical."""
    lib = emu.lib
    lib.emu_lsh_create.restype = ctypes.c_void_p
    lib.emu_lsh_query_count.restype = ctypes.c_int64
    rs = np.random.RandomState(6)
    k, b, r, n = 32, 8, 4, 600
    sig = rs.randint(0, 3, size=(n, k)).astype(np.uint32)          # low entropy: big buckets, many collisions
    sig[rs.randint(0, n, 80)] = sig[rs.randint(0, n, 80)]
    ref = o.DictLSH(k, b, r)
    for i, row in enumerate(sig):
        ref.insert(i, row.astype(np.uint64))
    h = ctypes.c_void_p(lib.emu_lsh_create(k, b, r, ctypes.c_int64(n + 10)))
    assert lib.emu_lsh_insert(h, _ptr(sig[:250]), ctypes.c_int64(250), 2) == 0          # two batches
    assert lib.emu_lsh_insert(h, _ptr(np.ascontiguousarray(sig[250:])), ctypes.c_int64(n - 250), 2) == 0
    q = np.ascontiguousarray(np.concatenate([sig[::3], rs.randint(0, 3, size=(40, k)).astype(np.uint32)]))
    nq = len(q)
    ptr = np.zeros(nq + 1, dtype=np.int64)
    total = lib.emu_lsh_query_count(h, _ptr(q), ctypes.c_int64(nq), _ptr(ptr), 2)
    assert total == ptr[-1] and ptr[0] == 0
    idx = np.full(max(total, 1), -1, dtype=np.int32)
    assert lib.emu_lsh_query_fill(h, _ptr(q), ctypes.c_int64(nq), _ptr(ptr), _ptr(idx), 2) == 0
    for j in range(nq):
        assert sorted(idx[ptr[j]:ptr[j + 1]].tolist()) == sorted(ref.query(q[j].astype(np.uint64))), j
    lib.emu_lsh_destroy(h)
    counts = rs.randint(0, 50, size=5000).astype(np.int64)
    out = np.zeros(5001, dtype=np.int64)
    assert lib.emu_exclusive_scan(_ptr(counts), ctypes.c_int64(5000), _ptr(out)) == 0
    assert np.array_equal(out, np.concatenate([[0], np.cumsum(counts)]))


def test_forest_query_kernel_vs_host_class(emu):
    """forest_query_kernel (warp-parallel binary search per tree, reference emission order) against this package's
    host MinHashLSHForest, which tests/test_lshforest.py pins to the reference's fixtures."""
    import datasketch_b200 as dsk
    lib = emu.lib
    rs = np.random.RandomState(4)
    for K, l in [(64, 4), (40, 40)]:
        n, kk = 500, K // l
        sig = rs.randint(0, 3, size=(n, K)).astype(np.uint32)
        sig[rs.randint(0, n, 60)] = sig[rs.randint(0, n, 60)]
        f = dsk.MinHashLSHForest(num_perm=K, l=l)
        for i, row in enumerate(sig):
            f.add(i, dsk.LeanMinHash(seed=1, hashvalues=row.astype(np.uint64)))
        f.index()
        order = np.stack([np.lexsort([np.arange(n)] + [sig[:, t * kk + c] for c in range(kk - 1, -1, -1)])
                          for t in range(l)]).astype(np.int32)
        q = np.ascontiguousarray(np.concatenate([sig[:40], rs.randint(0, 3, size=(10, K)).astype(np.uint32)]))
        for topk in (1, 7, 50):
            out = np.full((len(q), topk), -1, dtype=np.int32)
            assert lib.emu_forest_query(_ptr(sig), _ptr(order), ctypes.c_int64(n), K, l, kk, _ptr(q),
                                        ctypes.c_int64(len(q)), topk, _ptr(out), 1) == 0
            for j, row in enumerate(q):
                want = sorted(f.query(dsk.LeanMinHash(seed=1, hashvalues=row.astype(np.uint64)), topk))
                assert sorted(int(x) for x in out[j] if x >= 0) == want, (K, l, topk, j)


def test_jaccard_pairs_and_topk_kernels(emu):
    lib = emu.lib
    rs = np.random.RandomState(12)
    for k in (128, 100):
        n, m = 700, 900
        sig = rs.randint(0, 4, size=(n, k)).astype(np.uint32)
        ia, ib = rs.randint(0, n, size=m).astype(np.int64), rs.randint(0, n, size=m).astype(np.int64)
        cnt = np.zeros(m, dtype=np.int32)
        assert lib.emu_jaccard_pairs(_ptr(sig), ctypes.c_int64(n), k, _ptr(ia), _ptr(ib), ctypes.c_int64(m), _ptr(cnt)) == 0
        assert np.array_equal(cnt, (sig[ia] == sig[ib]).sum(axis=1))
    # top-k: smem-locked per-query lists, ties -> lower index, self excluded
    k, n, nq, topk, base = 64, 300, 70, 5, 100
    db = rs.randint(0, 3, size=(n, k)).astype(np.uint32)
    db[rs.randint(0, n, 20)] = db[rs.randint(0, n, 20)]
    q = np.ascontiguousarray(db[base:base + nq])
    oc_cnt = np.zeros((nq, topk), dtype=np.int32)
    oc_idx = np.zeros((nq, topk), dtype=np.int64)
    assert lib.emu_jaccard_topk(_ptr(q), ctypes.c_int64(nq), _ptr(db), ctypes.c_int64(n), k, topk, ctypes.c_int64(base),
                                _ptr(oc_cnt), _ptr(oc_idx), 1) == 0
    for i in range(nq):
        c = (db == q[i][None, :]).sum(axis=1).astype(np.int64)
        order = np.lexsort((np.arange(n), -c))
        order = order[order != base + i][:topk]
        assert np.array_equal(oc_idx[i], order) and np.array_equal(oc_cnt[i], c[order])


@pytest.mark.parametrize("k,n,nq,topk,vals", [(64, 200, 66, 5, 3), (128, 260, 40, 10, 1 << 32), (100, 257, 40, 7, 50), (32, 140, 10, 32, 2),
                                              (512, 140, 10, 10, 2), (1024, 140, 10, 32, 3)])
def test_topk_with_fingerprint_prefilter_equals_exact(emu, k, n, nq, topk, vals):
    """jaccard_topk_pf_kernel: bit-sliced 16-bit fingerprints give an upper bound of the match count; only pairs whose bound
    could still enter the list are counted exactly -- the lists must equal a brute-force ranking (and the exact kernel's):
    heavy ties (3 distinct values), no similarity at all (random 32-bit), K not a multiple of 32, topk = 32.  At K = 512 and
    1024 the prefilter's planes exceed a block's 227 KB of shared memory (the emulation enforces the limit): the launcher
    must run the exact kernel, whose footprint does not grow with K."""
    lib = emu.lib
    rs = np.random.RandomState(k + n)
    db = rs.randint(0, vals, size=(n, k), dtype=np.uint64).astype(np.uint32)
    db[rs.randint(0, n, 25)] = db[rs.randint(0, n, 25)]                # exact duplicates
    near = rs.randint(0, n, 40)
    db[near, : k // 2] = db[rs.randint(0, n, 40), : k // 2]             # half-equal rows
    base = 17
    q = np.ascontiguousarray(db[base:base + nq])
    for self_base in ((base, -1) if k == 64 else (base,)):     # "no self row" once; the emulated CTAs are slow
        got_c = np.zeros((nq, topk), dtype=np.int32)
        got_i = np.zeros((nq, topk), dtype=np.int64)
        assert lib.emu_jaccard_topk_pf(_ptr(q), ctypes.c_int64(nq), _ptr(db), ctypes.c_int64(n), k, topk,
                                       ctypes.c_int64(self_base), _ptr(got_c), _ptr(got_i), 1) == 0
        ex_c, ex_i = np.zeros_like(got_c), np.zeros_like(got_i)
        assert lib.emu_jaccard_topk(_ptr(q), ctypes.c_int64(nq), _ptr(db), ctypes.c_int64(n), k, topk,
                                    ctypes.c_int64(self_base), _ptr(ex_c), _ptr(ex_i), 1) == 0
        assert np.array_equal(got_c, ex_c) and np.array_equal(got_i, ex_i)
        for i in range(0, nq, 7):
            c = (db == q[i][None, :]).sum(axis=1).astype(np.int64)
            order = np.lexsort((np.arange(n), -c))
            if self_base >= 0:
                order = order[order != self_base + i]
            order = order[:topk]
            assert np.array_equal(got_i[i], order) and np.array_equal(got_c[i], c[order])


def test_sha1_kernel_vs_hashlib(emu):
    import hashlib
    import struct
    lib = emu.lib
    rs = np.random.RandomState(1)
    toks = [b"", b"a", b"abc", b"Hello", b"x" * 55, b"y" * 56, b"z" * 63, b"w" * 64, b"v" * 65, b"u" * 119, b"t" * 120,
            b"s" * 1000] + [bytes(rs.randint(0, 256, size=rs.randint(0, 200)).astype(np.uint8)) for _ in range(600)]
    blob = np.frombuffer(b"".join(toks) + b"\\0" * 8, dtype=np.uint8).copy()
    off = np.zeros(len(toks) + 1, dtype=np.int64)
    np.cumsum([len(t) for t in toks], out=off[1:])
    h32 = np.zeros(len(toks), dtype=np.uint32)
    h64 = np.zeros(len(toks), dtype=np.uint64)
    assert lib.emu_sha1_tokens(_ptr(blob), _ptr(off), ctypes.c_int64(len(toks)), _ptr(h32), 0) == 0
    assert lib.emu_sha1_tokens(_ptr(blob), _ptr(off), ctypes.c_int64(len(toks)), _ptr(h64), 1) == 0
    assert h32.tolist() == [struct.unpack("<I", hashlib.sha1(t).digest()[:4])[0] for t in toks]
    assert h64.tolist() == [struct.unpack("<Q", hashlib.sha1(t).digest()[:8])[0] for t in toks]


def test_xxh32_and_murmur3_kernels(emu, golden):
    """hash_tokens_kernel against the values the `xxhash` package produced (tests/golden/hashes.npz) and, for
    MurmurHash3, against the oracle restatement (itself pinned to published vectors in test_oracle_golden.py)."""
    lib = emu.lib
    g = golden("hashes")
    blob, off = np.ascontiguousarray(g["blob"]), np.ascontiguousarray(g["off"])
    n = len(off) - 1
    blob = np.concatenate([blob, np.zeros(8, np.uint8)])
    for seed in (0, 1, 0x9747B28C):
        out = np.zeros(n, dtype=np.uint32)
        assert lib.emu_hash_tokens(_ptr(blob), _ptr(off), ctypes.c_int64(n), 1, ctypes.c_uint32(seed), _ptr(out)) == 0
        assert np.array_equal(out, g[f"xxh32_seed{seed}"])
        assert lib.emu_hash_tokens(_ptr(blob), _ptr(off), ctypes.c_int64(n), 2, ctypes.c_uint32(seed), _ptr(out)) == 0
        want = [o.murmur3_32(bytes(blob[off[i]:off[i + 1]]), seed) for i in range(n)]
        assert out.tolist() == want


@pytest.mark.parametrize("tag", ["small", "tiny"])
def test_wmh_kernel_both_formulas(emu, golden, tag):
    """wmh_kernel<MANY = false / true> (host float32 ops, -ffp-contract=off) against the reference's fixtures."""
    lib = emu.lib
    for name, many in (("wmh", 0), ("wmh_many", 1)):
        g = golden(name)
        dim, ss, seed = (int(x) for x in g[f"{tag}_cfg"])
        rs_, ln_cs, betas = o.wmh_params(dim, ss, seed)
        cap = 6                                   # vectors per case: the emulation runs one host thread per CUDA thread
        V = np.ascontiguousarray(g[f"{tag}_X" if many else f"{tag}_v"], dtype=np.float32)
        V = np.ascontiguousarray(V[:cap])
        out = np.zeros((len(V), ss, 2), dtype=np.int64)
        status = np.zeros(len(V), dtype=np.int32)
        assert lib.emu_wmh(_ptr(np.ascontiguousarray(rs_)), _ptr(np.ascontiguousarray(ln_cs)), _ptr(np.ascontiguousarray(betas)),
                           ss, dim, _ptr(V), ctypes.c_int64(len(V)), _ptr(out), _ptr(status), many) == 0
        want = g[f"{tag}_out"][:len(V)]
        if many:
            null = g[f"{tag}_null"][:len(V)]
            assert np.array_equal(status.astype(bool), null)
            assert np.array_equal(out[~null], want[~null])
        else:
            assert not status.any() and np.array_equal(out, want)


# ---- randomised differential run ---------------------------------------------------------------------------------------
def _fuzz_signature_kernel(run, seed, iterations):
    """Random num_perm / document shapes / token kinds / modes / re-scan variants / init forms / unit and grid sizes;
    every case must equal the C oracle.  Returns the number of cases run."""
    rs = np.random.RandomState(seed)
    for it in range(iterations):
        k = int(rs.choice([1, 2, 7, 16, 31, 32, 33, 64, 65, 100, 128, 129, 192, 200, 256, 257, 300, 512, 520]))
        n = int(rs.randint(1, 40))
        style = int(rs.randint(0, 5))
        if style == 0:
            lens = rs.randint(0, 40, size=n)
        elif style == 1:
            lens = rs.randint(0, 600, size=n)
        elif style == 2:
            lens = np.where(rs.uniform(size=n) < 0.2, rs.randint(1500, 5000, size=n), rs.randint(0, 30, size=n))
        elif style == 3:
            lens = np.full(n, int(rs.choice([1, 15, 16, 17, 31, 32, 33, 512, 513])))
        else:
            lens = rs.randint(0, 3, size=n)
        off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lens, out=off[1:])
        T = int(off[-1])
        is64 = rs.uniform() < 0.15
        if is64:
            tok = rs.randint(0, 1 << 63, size=T + 1, dtype=np.uint64)[:T] * np.uint64(2) + rs.randint(0, 2, size=T).astype(np.uint64)
            mode = EXACT
        else:
            tok = rs.randint(0, 1 << 32, size=T + 1, dtype=np.uint64).astype(np.uint32)[:T]
            if rs.uniform() < 0.3 and T > 2:                                   # repeated tokens
                rep = np.nonzero(rs.uniform(size=T) < rs.uniform())[0]
                rep = rep[rep > 0]
                tok[rep] = tok[(rs.uniform(size=len(rep)) * rep).astype(np.int64)]
            if rs.uniform() < 0.2 and T > 0:                                   # tiny values: products next to the wrap
                tok[:T // 2] = rs.randint(0, 20, size=T // 2)
            mode = int(rs.randint(0, 3))
        perms = o.init_permutations(k, int(rs.randint(1, 50)))
        v1 = int(rs.randint(0, 2)) if mode == TWO_PHASE else 0
        init, u = None, rs.uniform()
        if u < 0.2:
            init = rs.randint(0, 1 << 32, size=k, dtype=np.uint64)
        elif u < 0.35:
            init = rs.randint(0, 1 << 32, size=(n, k), dtype=np.uint64).astype(np.uint32)
        elif u < 0.45:
            init = rs.randint(0, 1 << 32, size=(n, k), dtype=np.uint64)
        want = (oc.minhash_bulk_u64tok(tok, off, perms) if is64 else oc.minhash_bulk_u32tok(tok, off, perms)).astype(np.uint64)
        if init is not None:
            want = np.minimum(want, init.astype(np.uint64) if init.ndim == 2 else init.astype(np.uint64)[None, :])
        got = run(tok, off, perms, mode, v1=v1, init=init, out_u64=bool(rs.randint(0, 2)),
                  docs_per_unit=int(rs.choice([1, 2, 3, 7, 32])), grid_x=int(rs.randint(1, 3)))
        assert np.array_equal(got.astype(np.uint64), want), dict(seed=seed, it=it, k=k, n=n, style=style, is64=bool(is64),
                                                                 mode=mode, v1=v1, tokens=T)
    return iterations


def test_randomised_differential_vs_oracle(emu):
    """A slice of the fuzz run (10 000+ cases were run when this was written: no mismatch)."""
    assert _fuzz_signature_kernel(emu, seed=20260922, iterations=120) == 120



# ---- general variants of the signature kernel (GEN = 1: u32 tokens + any permutations, GEN = 2: u64 tokens) ----------
P61 = (1 << 61) - 1


def _unsafe_perms(k, rs):
    """Permutations built so that small 32-bit tokens land in the 36-value set where `% (2^61-1)` takes its conditional
    subtract (x = (j << 61) | lo with lo in [p - j, p]), mixed with seed-generated ones."""
    perms = o.init_permutations(k, 6).copy()
    for i in range(0, k, 3):
        j = int(rs.randint(0, 8))
        a = int(rs.choice([1, 3, 5, 1 << 20, (1 << 40) + 1]))
        h = int(rs.randint(0, 200))
        x = (j << 61) | (P61 - int(rs.randint(0, j + 1)))
        perms[0, i] = a
        perms[1, i] = (x - a * h) % (1 << 64)          # token h hits the subtract set for this permutation
    return perms


def _brute(tok, off, perms):
    """Python big-int restatement of minhash.py:294-297 for any permutations / 64-bit tokens (small inputs only)."""
    k = perms.shape[1]
    out = np.full((len(off) - 1, k), 0xFFFFFFFF, dtype=np.uint64)
    a = [int(v) for v in perms[0]]
    b = [int(v) for v in perms[1]]
    for d in range(len(off) - 1):
        for t in tok[int(off[d]):int(off[d + 1])]:
            t = int(t)
            for j in range(k):
                r = (((a[j] * t + b[j]) % (1 << 64)) % P61) & 0xFFFFFFFF
                if r < out[d, j]:
                    out[d, j] = r
    return out.astype(np.uint32)


@pytest.mark.parametrize("k", [16, 128, 192])
def test_general_u32_variant_with_unsafe_permutations(emu, k):
    rs = np.random.RandomState(100 + k)
    perms = _unsafe_perms(k, rs)
    lens = rs.randint(0, 60, size=24)
    lens[:3] = [0, 1, 17]
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rs.randint(0, 200, size=int(off[-1]), dtype=np.uint64).astype(np.uint32)     # small tokens: the subtract set is hit
    tok[::7] = rs.randint(0, 1 << 32, size=len(tok[::7]), dtype=np.uint64).astype(np.uint32)
    want = _brute(tok, off, perms)
    # the inputs really exercise the conditional subtract
    hit = 0
    for j in range(0, k, 3):
        for t in np.unique(tok):
            x = (int(perms[0, j]) * int(t) + int(perms[1, j])) % (1 << 64)
            hit += ((x & P61) + (x >> 61)) >= P61
    assert hit > 0
    assert np.array_equal(oc.minhash_bulk_u32tok(tok, off, perms), want)       # the C oracle agrees with the big-int form
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE, gen=1), want)
    assert np.array_equal(emu(tok, off, perms, EXACT), want)
    # and on ordinary input the general variant equals the default one
    tok2, off2 = _ragged(rs, 40, 300, extra_tail=2)
    safe = o.init_permutations(k, 1)
    assert np.array_equal(emu(tok2, off2, safe, TWO_PHASE, gen=1), oc.minhash_bulk_u32tok(tok2, off2, safe))


@pytest.mark.parametrize("k", [64, 128, 256, 300])
def test_u64_tokens_two_phase(emu, k):
    """GEN = 2: 64-bit hash values (minhash.py:294 accepts anything below 2^64).  Ragged documents, the <16-byte array tail
    (odd token count), units of several sizes, tokens that share their LOW word (phase 1 sees a tie, the exact stage must
    tell them apart), tiny / huge values, the de-duplication table's empty marker 2^64-1 as a token."""
    rs = np.random.RandomState(k)
    _, off = _ragged(rs, 50, 330, extra_tail=1)
    n = int(off[-1])
    tok = rs.randint(0, 1 << 63, size=n, dtype=np.uint64) * np.uint64(2) + rs.randint(0, 2, size=n, dtype=np.uint64)
    for d in range(0, len(off) - 1, 4):        # same low word, different high words
        a, b = int(off[d]), int(off[d + 1])
        if b - a > 8:
            tok[a + 1:a + 5] = (tok[a] & np.uint64(0xFFFFFFFF)) | (rs.randint(0, 1 << 32, size=4, dtype=np.uint64) << np.uint64(32))
    big = int(np.argmax(np.diff(off) >= 3))
    tok[int(off[big]):int(off[big]) + 3] = np.array([0, 1, 0xFFFFFFFFFFFFFFFF], dtype=np.uint64)
    perms = o.init_permutations(k, 5)
    want = oc.minhash_bulk_u64tok(tok, off, perms)
    for dpu, gx in ((3, 1), (32, 2), (1, 2)):
        assert np.array_equal(emu(tok, off, perms, TWO_PHASE, docs_per_unit=dpu, grid_x=gx), want), (k, dpu, gx)
    assert np.array_equal(emu(tok, off, perms, EXACT), want)
    # running-state merge and u64 output
    init = rs.randint(0, 1 << 32, size=want.shape, dtype=np.uint64)
    got = emu(tok, off, perms, TWO_PHASE, init=init, out_u64=True)
    assert got.dtype == np.uint64 and np.array_equal(got, np.minimum(want.astype(np.uint64), init))


def test_u64_tokens_small_against_big_int_form_and_unsafe_permutations(emu):
    rs = np.random.RandomState(3)
    k = 32
    perms = _unsafe_perms(k, rs)
    lens = np.array([0, 5, 40, 16, 1, 33], dtype=np.int64)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rs.randint(0, 200, size=int(off[-1]), dtype=np.uint64)
    tok[::3] = rs.randint(0, 1 << 63, size=len(tok[::3]), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    want = _brute(tok, off, perms)
    assert np.array_equal(oc.minhash_bulk_u64tok(tok, off, perms), want)
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE), want)


def test_u64_tokens_repeats_switch_deduplication_on(emu):
    """Heavy repetition of 64-bit tokens: flagged permutations -> de-duplicating staging on the 64-bit table -> off again."""
    rs = np.random.RandomState(5)
    lens = [200] * 3 + [256] * 8 + [130] * 40 + [250] * 4 + [700]
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rs.randint(0, 1 << 63, size=int(off[-1]), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    for d in list(range(3, 11)) + list(range(51, 56)):
        a, b = int(off[d]), int(off[d + 1])
        pool = tok[a:a + max(8, (b - a) // 4)].copy()
        pool[0] = np.uint64(0xFFFFFFFFFFFFFFFF)
        pool[1] = pool[2] ^ np.uint64(1 << 40)                 # equal low words, different tokens
        tok[a:b] = pool[rs.randint(0, len(pool), size=b - a)]
    perms = o.init_permutations(128, 9)
    want = oc.minhash_bulk_u64tok(tok, off, perms)
    emu.stats()
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE, docs_per_unit=64, grid_x=1), want)
    st = emu.stats()
    assert st["in_place"] == 0 and st["flagged"] >= 8 and st["removed"] > 300 and st["deduped"] >= 8 and st["copied"] >= 20, st
    assert np.array_equal(emu(tok, off, perms, TWO_PHASE, docs_per_unit=5, grid_x=2), want)


@pytest.mark.parametrize("gen", [1, 2])
def test_general_variants_long_documents_in_pieces(emu, gen):
    lib = emu.lib
    k = 128
    rs = np.random.RandomState(40 + gen)
    lens = np.array([30, 250, 0, 101, 100, 1000, 7, 99, 481, 40, 2100, 12], dtype=np.int64)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    if gen == 2:
        tok = rs.randint(0, 1 << 63, size=int(off[-1]), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
        perms = o.init_permutations(k, 4)
        want = oc.minhash_bulk_u64tok(tok, off, perms)
    else:
        tok = rs.randint(0, 1 << 32, size=int(off[-1]), dtype=np.uint64).astype(np.uint32)
        perms = _unsafe_perms(k, rs)
        tok[::5] = rs.randint(0, 200, size=len(tok[::5]))
        want = oc.minhash_bulk_u32tok(tok, off, perms)
    a, b = np.ascontiguousarray(perms[0]), np.ascontiguousarray(perms[1])
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.emu_minhash_sig_long.argtypes = [vp, vp, i64, vp, vp, ci, vp, i64, ci, vp, ci, ci, ci, i64, ci, vp, ci]
    n = len(lens)
    for dpu, gx in ((3, 1), (32, 2)):
        out = np.zeros((n, k), dtype=np.uint32)
        assert lib.emu_minhash_sig_long(tok.ctypes.data, off.ctypes.data, n, a.ctypes.data, b.ctypes.data, k, None, 0, 0,
                                        out.ctypes.data, 0, dpu, gx, 100, 5, None, gen) == 0
        assert np.array_equal(out, want), (gen, dpu, gx)


@pytest.mark.parametrize("k,b,r", [(128, 32, 4), (256, 17, 15), (64, 9, 7), (16, 4, 4)])
def test_fused_lsh_insert_from_tokens_vs_dict_oracle(emu, k, b, r):
    """signature_kernel.cu template LSH (dsk_lsh_insert_tokens' fused route): the warp that finishes a document inserts
    it.  Token lists with planted near-duplicates and exact duplicates (so buckets have several members and chains get
    contended), empty and ragged documents, two batches (the second one lands behind the first in the index), several
    unit sizes; afterwards the index's rows equal the oracle's signatures and every query's candidate set equals the
    reference's dict buckets (oracle DictLSH = lsh.py:326-347, :370-432)."""
    lib = emu.lib
    lib.emu_lsh_create.restype = ctypes.c_void_p
    lib.emu_lsh_query_count.restype = ctypes.c_int64
    lib.emu_lsh_rows.restype = ctypes.c_void_p
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.emu_lsh_insert_tokens.argtypes = [vp, vp, vp, i64, vp, vp, ci, ci, ci]
    rs = np.random.RandomState(k + b)
    n = 150
    docs = []
    for i in range(n):
        if i % 5 == 3 and i > 10:                       # near-duplicate of an earlier document: a few tokens resampled
            base = docs[int(rs.randint(0, i))].copy()
            if len(base):
                base[rs.randint(0, len(base), size=max(1, len(base) // 40))] = rs.randint(0, 1 << 32, dtype=np.uint64)
            docs.append(base)
        elif i % 11 == 7:
            docs.append(docs[i - 1].copy())             # exact duplicate
        else:
            docs.append(rs.randint(0, 1 << 32, size=int(rs.choice([0, 3, 40, 64, 130, 256, 300])), dtype=np.uint64).astype(np.uint32))
    docs = [np.asarray(d, dtype=np.uint32) for d in docs]
    perms = o.init_permutations(k, 2)
    a, bb = np.ascontiguousarray(perms[0]), np.ascontiguousarray(perms[1])
    ref = o.DictLSH(k, b, r)
    want_rows = []
    h = ctypes.c_void_p(lib.emu_lsh_create(k, b, r, ctypes.c_int64(n + 5)))
    for (lo, hi), (dpu, gx) in zip(((0, 60), (60, n)), ((3, 1), (32, 2))):
        part = docs[lo:hi]
        off = np.zeros(len(part) + 1, dtype=np.int64)
        np.cumsum([len(d) for d in part], out=off[1:])
        tok = np.concatenate(part + [np.zeros(4, np.uint32)])[:int(off[-1])]
        tok = np.ascontiguousarray(tok)
        sig = oc.minhash_bulk_u32tok(tok, off, perms)
        want_rows.append(sig)
        for i, row in enumerate(sig):
            ref.insert(lo + i, row.astype(np.uint64))
        assert lib.emu_lsh_insert_tokens(h, tok.ctypes.data, off.ctypes.data, len(part), a.ctypes.data, bb.ctypes.data, k, dpu, gx) == 0
    want_rows = np.concatenate(want_rows)
    rows = np.ctypeslib.as_array(ctypes.cast(lib.emu_lsh_rows(h), ctypes.POINTER(ctypes.c_uint32)), shape=(n + 5, k))[:n]
    assert np.array_equal(rows, want_rows)
    q = np.ascontiguousarray(want_rows[::2])
    nq = len(q)
    ptr = np.zeros(nq + 1, dtype=np.int64)
    total = lib.emu_lsh_query_count(h, _ptr(q), ctypes.c_int64(nq), _ptr(ptr), 2)
    idx = np.full(max(total, 1), -1, dtype=np.int32)
    assert lib.emu_lsh_query_fill(h, _ptr(q), ctypes.c_int64(nq), _ptr(ptr), _ptr(idx), 2) == 0
    multi = 0
    for j in range(nq):
        got = sorted(idx[ptr[j]:ptr[j + 1]].tolist())
        assert got == sorted(ref.query(q[j].astype(np.uint64))), j
        multi += len(got) > 1
    assert multi >= 5            # the planted duplicates really share buckets
    lib.emu_lsh_destroy(h)


@pytest.mark.parametrize("gen", [1, 2])
def test_general_variants_structured_tokens_wraps_and_extreme_parameters(emu, gen):
    """The general variants on the inputs random data never produces: tiny and near-2^32 low words (L' < 8: the wrap of
    L' - 8, many exact ties), high words 0 / 1 / 2^32-1, tokens 0 and 2^64-1, and permutations at the ends of their ranges
    (a = 1, a = p - 1, b = 0, b = p - 1, a with a zero low word) next to ones built to hit the conditional subtract."""
    rs = np.random.RandomState(gen)
    lo = np.concatenate([np.arange(0, 1500, dtype=np.uint64), np.uint64(1 << 32) - np.arange(1, 1501, dtype=np.uint64),
                         np.zeros(250, dtype=np.uint64), np.full(250, 0xFFFFFFFF, dtype=np.uint64)])
    k = 64
    perms = _unsafe_perms(k, rs)
    perms[0, 1], perms[1, 1] = 1, 0
    perms[0, 2], perms[1, 2] = P61 - 1, P61 - 1
    perms[0, 4], perms[1, 4] = np.uint64(7 << 32), 5              # a_lo = 0: L' is the same for every token
    perms[0, 5], perms[1, 5] = 1, P61 - 1                          # x = h + p - 1: the subtract fires for h = 1 .. 8
    off = np.arange(0, len(lo) + 1, 125, dtype=np.int64)
    if gen == 2:
        hi = rs.choice(np.array([0, 1, 0xFFFFFFFF, 0x80000000, 12345], dtype=np.uint64), size=len(lo))
        tok = (hi << np.uint64(32)) | lo
        tok[7], tok[130] = np.uint64(0), np.uint64(0xFFFFFFFFFFFFFFFF)
        want = oc.minhash_bulk_u64tok(tok, off, perms)
        small = slice(0, 2)                         # the big-int form on the first two documents pins the C oracle here too
        assert np.array_equal(want[small], _brute(tok[:250], off[:3], perms))
        assert np.array_equal(emu(tok, off, perms, TWO_PHASE, docs_per_unit=5, grid_x=2), want)
    else:
        tok = lo.astype(np.uint32)
        want = oc.minhash_bulk_u32tok(tok, off, perms)
        assert np.array_equal(want[:2], _brute(tok[:250], off[:3], perms))
        assert np.array_equal(emu(tok, off, perms, TWO_PHASE, gen=1, docs_per_unit=5, grid_x=2), want)
    assert np.array_equal(emu(tok, off, perms, EXACT), want)
