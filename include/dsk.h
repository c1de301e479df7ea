/* dsk.h -- C-ABI of libdsk_b200.so: the B200 (sm_100a) MinHash / LSH signature engine.
 *
 * The reference (ekzhu/datasketch 1.10.0) is pure Python and exposes NO plugin /
 * FFI interface; its only backend seam is the `gpu_mode` switch inside
 * MinHash.update_batch (datasketch/minhash.py:117, :270-291).  This header is the
 * boundary a maintainer would bind with ctypes to replace that seam and the
 * Python loops around it (see INTEGRATION.md for the stub).  Each entry point
 * cites the reference code it replaces.
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures (streams are void*,
 *     i.e. a cudaStream_t / CUstream value; NULL = the legacy default stream).
 *   - "d_" parameters are DEVICE pointers owned by the caller (e.g. torch tensors'
 *     data_ptr()); "h_" parameters are HOST pointers.
 *   - device entry points are stream-ordered and asynchronous; return 0 when the
 *     work was enqueued, non-zero DSK_ERR_* otherwise; dsk_last_error() returns a
 *     thread-local message for the last failure on the calling thread.
 *   - integer results are bit-exact with the reference's numpy uint64 path.
 */
#ifndef DSK_H_
#define DSK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSK_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define DSK_API __attribute__((visibility("default")))
#else
#define DSK_API
#endif

enum {
    DSK_OK = 0,
    DSK_ERR_INVALID = 1,   /* bad argument (maps to ValueError in the Python host layer) */
    DSK_ERR_CUDA = 2,      /* CUDA runtime error (maps to RuntimeError) */
    DSK_ERR_NO_DEVICE = 3, /* no sm_100 device: there is NO CPU fallback (RuntimeError) */
    DSK_ERR_ALIGN = 4,     /* pointer alignment contract violated */
    DSK_ERR_NOMEM = 5
};

/* kernel selection for dsk_minhash_bulk (flags) */
enum {
    DSK_KERNEL_AUTO = 0,     /* = TWO_PHASE */
    DSK_KERNEL_TWO_PHASE = 1,/* the two-phase signature kernel; bit-exact for ANY permutation and u32 / u64 tokens: the default
                                variant needs 32-bit tokens and n_unsafe == 0, otherwise a general variant runs that
                                takes the conditional subtract of `% (2^61-1)` in its exact stage (window 8 instead of 7) */
    DSK_KERNEL_DIRECT = 2,   /* r = lo32(x) + top3(x) per (token, perm), no candidate filtering; DSK_ERR_INVALID unless
                                the tokens are 32-bit and n_unsafe == 0 */
    DSK_KERNEL_EXACT = 3     /* full 64-bit `% (2^61-1)` per evaluation; any permutation, u32/u64 tokens (round 1's kernel) */
};

DSK_API int dsk_version(void);
DSK_API const char *dsk_last_error(void);

/* Number of usable CUDA devices; *sm_count / *cc receive properties of `device`.
 * Replaces datasketch/minhash.py:38-48 (_gpu_available). */
DSK_API int dsk_device_count(void);
DSK_API int dsk_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem);

/* ---- permutation handle -------------------------------------------------------
 * Uploads the (a, b) parameters of MinHash._init_permutations
 * (datasketch/minhash.py:170-184; generated on the HOST with numpy, never on
 * device) and analyses them once: `n_unsafe` = number of permutations for which
 * some 32-bit token value h makes ((a*h+b) mod 2^64) fall in the 36-value set
 * where `% (2^61-1)` needs its conditional subtract.  n_unsafe == 0 (true for every seed-generated
 * set tested) selects the two-phase kernel's default variant and allows DSK_KERNEL_DIRECT; otherwise the
 * two-phase kernel's general variant runs (same speed class, still bit-exact).
 * Replaces minhash.py:160-165 (_ensure_gpu_caches). */
typedef struct dsk_perm dsk_perm;
DSK_API int dsk_perm_create(const uint64_t *h_a, const uint64_t *h_b, int num_perm, int device, dsk_perm **out);
DSK_API int dsk_perm_info(const dsk_perm *p, int *num_perm, int *n_unsafe, int *device);
DSK_API void dsk_perm_destroy(dsk_perm *p);
/* Host-only analysis (no device needed): out_unsafe[i] = 1 iff permutation i can reach the
 * conditional-subtract set with some token h < 2^32.  Returns the number of unsafe ones. */
DSK_API int dsk_perm_analyze(const uint64_t *h_a, const uint64_t *h_b, int num_perm, uint8_t *out_unsafe);

/* ---- bulk signature build -------------------------------------------------------
 * Replaces MinHash.update_batch's hot loop (datasketch/minhash.py:294-297 CPU,
 * :281-291 CuPy) batched over documents as in MinHash.bulk / generator
 * (:464-522): for document i with token hashes tokens[offsets[i]:offsets[i+1]],
 *   out[i][k] = min(init[i][k], min_t (((a_k*h_t + b_k) mod 2^64) % (2^61-1)) & 0xFFFFFFFF)
 * d_tokens   u32 (token_is_u64=0) or u64 (=1) token hashes, 16-byte aligned
 * d_offsets  int64[n_docs+1], non-decreasing CSR offsets, offsets[n_docs] == n_tokens
 * d_init     NULL (empty state, all 0xFFFFFFFF: minhash.py:167-168) or running
 *            signatures to merge (update_batch on a non-empty MinHash, :297);
 *            init_stride = elements between rows (0 = one row broadcast to all docs)
 * d_out      [n_docs, num_perm] u32 (out_is_u64=0) or u64 (=1; the reference's dtype)
 * flags      DSK_KERNEL_*  */
DSK_API int dsk_minhash_bulk(const dsk_perm *perm, const void *d_tokens, int token_is_u64,
                     const int64_t *d_offsets, int64_t n_docs, int64_t n_tokens,
                     const void *d_init, int64_t init_stride, int init_is_u64,
                     void *d_out, int out_is_u64, int flags, void *stream);

/* Same, with a caller-provided device workspace that lets the library cut LONG documents (> 4096 tokens) into pieces
 * of 1024 tokens on the device: the warp that meets such a document stores the row's initial value and appends the
 * pieces to a table in the workspace; a second launch spreads the pieces over all warps and min-merges their partial
 * signatures into the row (atomicMin; MinHash.merge is the combine rule, minhash.py:337-359).  Without a workspace
 * (dsk_minhash_bulk) one warp handles a whole document, whatever its length.  d_workspace: 16-byte aligned,
 * >= dsk_minhash_bulk_workspace_size(n_docs, n_tokens) bytes (0 when no document can be long), contents undefined on
 * entry and on return, owned by the caller, in use until the launch has finished on `stream`.
 * The reference's own GPU benchmark shape is one 50 000-token update_batch (benchmark/sketches/minhash_gpu_benchmark.py:42-48). */
DSK_API size_t dsk_minhash_bulk_workspace_size(int64_t n_docs, int64_t n_tokens);
DSK_API int dsk_minhash_bulk_ws(const dsk_perm *perm, const void *d_tokens, int token_is_u64,
                        const int64_t *d_offsets, int64_t n_docs, int64_t n_tokens,
                        const void *d_init, int64_t init_stride, int init_is_u64,
                        void *d_out, int out_is_u64, int flags, void *d_workspace, size_t workspace_bytes, void *stream);

/* Fused signature build + all-gather (multi-GPU): like dsk_minhash_bulk, but each signature row
 * is stored straight into row (row_offset + i) of the FULL [N_total, num_perm] matrix of every
 * rank: h_peer_out[0..n_peers) are device pointers to those matrices (this rank's own buffer
 * and its peers' buffers mapped over NVLink, e.g. torch symmetric memory / cudaIpc).  The
 * transfer overlaps the integer math document by document; the caller synchronises the ranks
 * afterwards (stream sync + barrier).  Replaces "build, then ncclAllGather". */
DSK_API int dsk_minhash_bulk_gather(const dsk_perm *perm, const void *d_tokens, int token_is_u64,
                                    const int64_t *d_offsets, int64_t n_docs, int64_t n_tokens,
                                    void *const *h_peer_out, int n_peers, int64_t row_offset,
                                    int out_is_u64, int flags, void *stream);

/* Host-buffer variant: same computation, tokens/offsets/out are HOST pointers
 * (pinned memory gives full PCIe overlap; pageable memory is staged).  Documents
 * are cut into slices and H2D copy, kernel and D2H copy are pipelined over
 * internal streams; returns after the last slice landed in h_out.
 * This is the call the reference-facing MinHash.bulk makes. */
DSK_API int dsk_minhash_bulk_host(const dsk_perm *perm, const void *h_tokens, int token_is_u64,
                          const int64_t *h_offsets, int64_t n_docs,
                          const void *h_init, int64_t init_stride, int init_is_u64,
                          void *h_out, int out_is_u64, int flags);

/* Ownership (see INTEGRATION.md "What the library allocates"): every d_ / h_ buffer above is the caller's.  The
 * library itself holds (a) per dsk_perm handle: the permutation table, 16 KB of work counters and 64 events, freed by
 * dsk_perm_destroy; (b) per device, created by the first dsk_minhash_bulk_host call and grown on demand: three
 * streams and three slots of device + pinned staging buffers sized to the largest slice seen (<= 16 Mi tokens,
 * <= 128 Ki documents per slice).  dsk_release_host_pipeline frees (b) for `device` (-1 = every device); the next
 * host-buffer call re-creates it.  Not to be called concurrently with dsk_minhash_bulk_host on the same device. */
DSK_API int dsk_release_host_pipeline(int device);

/* Element-wise min of two signature matrices (MinHash.merge / union,
 * datasketch/minhash.py:359, :453; LeanMinHash.union lean_minhash.py:249). */
DSK_API int dsk_sig_merge_min(const uint32_t *d_x, const uint32_t *d_y, int64_t n_elems, uint32_t *d_out, void *stream);

/* ---- signature codecs (HBM-bound) ---------------------------------------------------
 * LeanMinHash records: `struct` layout "<bo> q i {K}I" = seed int64, K int32, K x uint32
 * (datasketch/lean_minhash.py:174-175 serialize, :201-214 deserialize, :216-232 pickle
 * state).  big_endian = 0 for byteorder '<' '=' '@' (x86-64: 12 + 4K bytes, no padding),
 * 1 for '>' '!'.  d_rec is [n, 12 + 4K] bytes.  Unpack validates every header against
 * (seed, K) and sets *d_status = 1 on a mismatch (d_status must be zeroed by the caller). */
DSK_API int dsk_lean_pack(const void *d_sig, int sig_is_u64, int64_t n, int num_perm, int64_t seed, int big_endian,
                          uint8_t *d_rec, void *stream);
DSK_API int dsk_lean_unpack(const uint8_t *d_rec, int64_t n, int num_perm, int64_t seed, int big_endian, void *d_sig,
                            int sig_is_u64, int *d_status, void *stream);

/* MinHashLSH band keys: for document i and band j, the r hash values
 * sig[i][j*r:(j+1)*r] as big-endian uint64 -- byte-identical to the reference's default
 * `_H` = bytes(hashvalues[start:end].byteswap().data) (datasketch/lsh.py:344, :427, :537-538).
 * d_keys is [n, b, 8*r] bytes. */
DSK_API int dsk_band_keys(const uint32_t *d_sig, int64_t n, int num_perm, int b, int r, uint8_t *d_keys, void *stream);

/* 64-bit fingerprint of each band's r-tuple, [n, b] uint64: the bucket key of the GPU LSH
 * index (equal tuples <=> equal fingerprints up to hash collisions, which the LSH kernels
 * resolve by comparing the tuples themselves). */
DSK_API int dsk_band_fingerprints(const uint32_t *d_sig, int64_t n, int num_perm, int b, int r, uint64_t *d_fp,
                                  void *stream);

/* ---- MinHashLSHBloom ("next" row, SURVEY.md 8f rank 3) -----------------------------------------------
 * dsk_band_sums: the Bloom key of every band, d_keys[i][j] = sum(sig[i][j*r:(j+1)*r]) % (2^61 - 1) as uint64
 * ([n, b]) -- BloomTable.insert / query's `x = sum(hashvalues) % _mersenne_prime`
 * (datasketch/lsh_bloom.py:94-106, :108-118, :20).  HBM-bound codec: 4*num_perm bytes in, 8*b out per document.
 * dsk_bloom_insert / dsk_bloom_query: the same keys go straight into / are tested against b device-resident
 * Bloom tables (MinHashLSHBloom._insert :308-316, query :365-371: a hit in ANY band flags the document).
 * d_bits is [b][words_per_table] uint32, caller-owned and zero-initialised; each key sets / tests n_hashes
 * bits among the table's first n_bits bits (double hashing).  The reference delegates the bit tables to
 * pybloomfilter; these are the library's own (no false negatives, the usual (1 - e^(-kn/m))^k false-positive
 * rate), not pybloomfilter's file format.  d_hit is [n] uint8 (1 = duplicate candidate). */
DSK_API int dsk_band_sums(const uint32_t *d_sig, int64_t n, int num_perm, int b, int r, uint64_t *d_keys, void *stream);
DSK_API int dsk_bloom_insert(const uint32_t *d_sig, int64_t n, int num_perm, int b, int r, uint32_t *d_bits,
                             uint64_t words_per_table, uint64_t n_bits, int n_hashes, void *stream);
DSK_API int dsk_bloom_query(const uint32_t *d_sig, int64_t n, int num_perm, int b, int r, const uint32_t *d_bits,
                            uint64_t words_per_table, uint64_t n_bits, int n_hashes, uint8_t *d_hit, void *stream);

/* ---- Weighted MinHash (Ioffe ICWS) ------------------------------------------------------
 * Handle = device copy of the generator parameters rs, ln_cs, betas, each [sample_size, dim]
 * float32, drawn on the HOST by numpy exactly as WeightedMinHashGenerator.__init__ does
 * (datasketch/weighted_minhash.py:118-121).  dsk_wmh_minhash replaces the per-sample loop
 * of WeightedMinHashGenerator.minhash (:147-158) for a batch of n vectors:
 *   d_v      [n, dim] float32 weights (zeros are skipped, :148-152)
 *   d_out    [n, sample_size, 2] int64: (k, int(t_k)) per sample (:158)
 *   d_status [n] int32: 1 where the input row is all zeros (reference: ValueError, :149-150)
 *   flags    DSK_WMH_MINHASH (0), or DSK_WMH_MINHASH_MANY: the float32 operation order of the
 *            reference's experimental minhash_many (:221-224; an all-zero row is None there, :241-245)
 *            | DSK_WMH_INPUT_LOG: d_v holds ln(weight) already (float32, NaN where the weight is zero) -- the host
 *            layer passes numpy's own float32 log (:152), which makes every step bit-identical to the reference;
 *            without it the kernel takes a correctly rounded log itself (<= 1 ulp from numpy's) */
#define DSK_WMH_MINHASH 0
#define DSK_WMH_MINHASH_MANY 1
#define DSK_WMH_INPUT_LOG 2
typedef struct dsk_wmh dsk_wmh;
DSK_API int dsk_wmh_create(const float *h_rs, const float *h_ln_cs, const float *h_betas, int sample_size, int dim,
                           int device, dsk_wmh **out);
DSK_API void dsk_wmh_destroy(dsk_wmh *g);
DSK_API int dsk_wmh_minhash(const dsk_wmh *g, const float *d_v, int64_t n, int64_t *d_out, int32_t *d_status,
                            int flags, void *stream);

/* ---- device-resident MinHashLSH index ------------------------------------------------------
 * Replaces the bucket step of MinHashLSH._insert / query over dict storage
 * (datasketch/lsh.py:344-347, :426-429; storage.py:209-259) for whole batches.  Documents are
 * numbered 0..n_docs-1 in insertion order (the host layer maps numbers to user keys).  Buckets
 * are exact: two documents meet iff a band's r-tuple is equal, as with the reference's byte keys.
 *   dsk_lsh_insert       append n signatures ([n, num_perm] u32) to the index
 *   dsk_lsh_insert_tokens  the same from TOKENS: builds the n documents' signatures (dsk_minhash_bulk's kernel) straight into
 *                        the index's own signature storage and inserts each document in the same launch -- the warp that
 *                        finishes a row does its b bucket updates, whose DRAM latency hides behind the other warps'
 *                        integer work; the signature matrix is never read back.  (MinHash.bulk + MinHashLSH.insert per
 *                        document, minhash.py:464-489 + lsh.py:326-347.)  Fused for u32 tokens, a handle with
 *                        n_unsafe == 0 and num_perm <= 256; any other input runs the two kernels one after the other.
 *   dsk_lsh_query_count  d_counts[q] = number of distinct candidates of query q
 *   dsk_exclusive_scan   d_out[0..n] = exclusive prefix sums of d_in[0..n-1] (d_out[n] = total);
 *                        d_scratch holds at least n/1024 + 2 int64
 *   dsk_lsh_query_fill   writes each query's candidates (document numbers, unordered like the
 *                        reference's list(set), lsh.py:432) at d_idx[d_ptr[q] .. d_ptr[q+1]) */
typedef struct dsk_lsh dsk_lsh;
DSK_API int dsk_lsh_create(int num_perm, int b, int r, int64_t capacity_docs, int device, dsk_lsh **out);
DSK_API void dsk_lsh_destroy(dsk_lsh *ix);
DSK_API int dsk_lsh_size(const dsk_lsh *ix, int64_t *n_docs, int64_t *capacity_docs);
DSK_API int dsk_lsh_insert(dsk_lsh *ix, const uint32_t *d_sig, int64_t n, void *stream);
DSK_API int dsk_lsh_insert_tokens(dsk_lsh *ix, const dsk_perm *perm, const void *d_tokens, int token_is_u64,
                                  const int64_t *d_offsets, int64_t n_docs, int64_t n_tokens, void *stream);
DSK_API int dsk_lsh_query_count(const dsk_lsh *ix, const uint32_t *d_qsig, int64_t nq, int64_t *d_counts, void *stream);
DSK_API int dsk_lsh_query_fill(const dsk_lsh *ix, const uint32_t *d_qsig, int64_t nq, const int64_t *d_ptr,
                               int32_t *d_idx, void *stream);
DSK_API int dsk_exclusive_scan(const int64_t *d_in, int64_t n, int64_t *d_out, int64_t *d_scratch, void *stream);

/* ---- Jaccard estimate -----------------------------------------------------------------------
 * d_count[p] = number of positions where rows d_i[p] and d_j[p] of the [n_rows, num_perm] u32
 * signature matrix are equal; jaccard = count / num_perm (MinHash.jaccard,
 * datasketch/minhash.py:324; seeds / lengths are validated by the host layer as :314-323).
 * An out-of-range pair index yields -1. */
DSK_API int dsk_jaccard_pairs(const uint32_t *d_sig, int64_t n_rows, int num_perm, const int64_t *d_i,
                              const int64_t *d_j, int64_t m, int32_t *d_count, void *stream);

/* All-pairs top-k: for each of nq query rows, the `topk` (<= 32) rows of the [n, num_perm]
 * (num_perm <= 4096) database with the most equal positions, best first; ties -> lower database index.  If
 * self_base >= 0, query i is database row self_base + i and is excluded from its own list.
 * d_cnt [nq, topk] int32 counts (jaccard = cnt / num_perm), d_idx [nq, topk] int64 (-1 pads). */
DSK_API int dsk_jaccard_topk(const uint32_t *d_q, int64_t nq, const uint32_t *d_db, int64_t n, int num_perm, int topk,
                             int64_t self_base, int32_t *d_cnt, int64_t *d_idx, void *stream);
/* Same result, ~3x fewer ALU ops: with a caller-provided workspace (16-byte aligned, >= dsk_jaccard_topk_workspace_size()
 * bytes -- 0 means the prefilter does not apply and the call behaves like dsk_jaccard_topk: num_perm < 32, num_perm > 480
 * (the fingerprint planes would not fit a block's shared memory) or n < 512) both matrices are first reduced
 * to bit-sliced 16-bit fingerprints; a pair reaches the exact count only if the fingerprint agreement -- an upper bound of
 * the number of equal positions -- could still enter the query's list.  Lists are identical to dsk_jaccard_topk's. */
DSK_API size_t dsk_jaccard_topk_workspace_size(int64_t nq, int64_t n, int num_perm);
DSK_API int dsk_jaccard_topk_ws(const uint32_t *d_q, int64_t nq, const uint32_t *d_db, int64_t n, int num_perm, int topk,
                                int64_t self_base, int32_t *d_cnt, int64_t *d_idx, void *d_workspace,
                                size_t workspace_bytes, void *stream);

/* ---- LSH Forest query ("next" row, SURVEY.md 8f) ----------------------------------------------
 * d_order is [l, n] int32: for tree t, the document numbers sorted by (sig[doc][t*k:(t+1)*k]
 * lexicographically, document number) -- the flattening of the reference's sorted key list +
 * insertion-ordered buckets (datasketch/lshforest.py:68-72).  For each query the kernel walks
 * prefix lengths r = k..1 and trees 0..l-1 exactly like MinHashLSHForest.query (:74-128) and writes
 * the first `topk` (<= 1024) distinct document numbers it meets (d_out [nq, topk], -1 pads). */
DSK_API int dsk_forest_query(const uint32_t *d_sig, const int32_t *d_order, int64_t n, int num_perm, int l, int k,
                             const uint32_t *d_qsig, int64_t nq, int topk, int32_t *d_out, void *stream);

/* ---- b-bit MinHash blocks ("next" row, SURVEY.md 8f) -----------------------------------------
 * bBitMinHash keeps the b lowest bits of each value (datasketch/b_bit_minhash.py:38) and packs
 * them into 64-bit blocks, value j of a block at bit (n-1-j)*slot with slot = 1,2,4,8,16,32 >= b
 * and n = 64/slot (:78-92).  d_blocks is [n, ceil(num_perm / n)] uint64 (the payload after the
 * 21-byte '<qBdi' header of the pickle state). */
DSK_API int dsk_bbit_pack(const uint32_t *d_sig, int64_t n, int num_perm, int b, uint64_t *d_blocks, void *stream);
DSK_API int dsk_bbit_unpack(const uint64_t *d_blocks, int64_t n, int num_perm, int b, uint32_t *d_sig, void *stream);

/* ---- default token hash on device ("next" row, SURVEY.md 8f) --------------------------------
 * d_out[t] = sha1_hash32 (out_is_u64 = 0) or sha1_hash64 (= 1) of the byte string
 * d_bytes[d_byte_offsets[t] : d_byte_offsets[t+1]] -- datasketch/hashfunc.py:5-28, i.e. the
 * first 4 / 8 bytes of SHA-1 read little-endian.  Lets MinHash.bulk with the default hashfunc
 * skip the per-token Python hashlib loop (minhash.py:263). */
DSK_API int dsk_sha1_tokens(const uint8_t *d_bytes, const int64_t *d_byte_offsets, int64_t n_tokens, void *d_out,
                            int out_is_u64, void *stream);

/* ---- fast non-cryptographic token hashes on device ("next" row, SURVEY.md 8f rank 1) -------------
 * The hash functions the reference documents as `hashfunc` alternatives (docs/minhash.rst:79-112):
 *   DSK_HASH_XXH32       XXH32(data, seed)             == xxhash.xxh32_intdigest(data, seed)
 *   DSK_HASH_MURMUR3_32  MurmurHash3_x86_32(data, seed) == mmh3.hash(data, seed, signed=False)
 * d_out[t] = 32-bit hash of d_bytes[d_byte_offsets[t] : d_byte_offsets[t+1]]; replaces the per-token
 * Python call of minhash.py:263 when the user's hashfunc is one of these. */
#define DSK_HASH_XXH32 1
#define DSK_HASH_MURMUR3_32 2
DSK_API int dsk_hash_tokens(const uint8_t *d_bytes, const int64_t *d_byte_offsets, int64_t n_tokens, int kind,
                            uint32_t seed, uint32_t *d_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DSK_H_ */
