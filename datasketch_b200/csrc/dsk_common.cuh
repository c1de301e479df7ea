// dsk_common.cuh -- shared device helpers (sm_100a): mbarrier / bulk-copy (TMA) PTX,
// error plumbing.  No torch, no libraries: plain CUDA runtime + inline PTX.
#pragma once
#ifdef DSK_EMU  // CPU emulation of the kernel logic for the test-suite (tests/emu/cuda_emu.h); never defined in the product build
#include "cuda_emu.h"
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/dsk.h"

// Kernel launch and dynamic shared memory go through two macros so that the CPU emulation used by the test-suite
// (tests/emu, -DDSK_EMU) can run the launchers' host logic too.  In the product build they expand to the plain CUDA forms.
#ifdef DSK_EMU
#define DSK_LAUNCH(kernel, grid, block, smem, stream, ...) ::emu_launch(kernel, grid, block, smem, __VA_ARGS__)
#define DSK_DYNAMIC_SMEM(name) unsigned char *name = ::emu_dynamic_smem()
#define DSK_DYNAMIC_SMEM_T(type, name, align) type *name = reinterpret_cast<type *>(::emu_dynamic_smem())
#else
#define DSK_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<grid, block, smem, stream>>>(__VA_ARGS__)
#define DSK_DYNAMIC_SMEM(name) extern __shared__ __align__(128) unsigned char name[]
#define DSK_DYNAMIC_SMEM_T(type, name, align) extern __shared__ __align__(align) type name[]
#endif

namespace dsk {

// dynamic shared memory one block may opt in to on sm_100 (227 KB); launchers size their tiles against it
constexpr size_t kMaxDynamicSmemPerBlock = 232448;

// ---- thread-local error string --------------------------------------------------
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);

#define DSK_CUDA(call)                                            \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) return ::dsk::cuda_fail(e__, #call); \
    } while (0)

// ---- parameters of the bulk signature kernels (minhash_kernels.cu) ----------------------
struct BulkParams {
    const void *tokens;         // u32 or u64 token hashes, 16-byte aligned
    const int64_t *offsets;     // [n_docs + 1] CSR offsets relative to `tokens`
    int64_t n_docs, n_tokens;
    const uint32_t *a_lo, *a_hi, *b_lo, *b_hi;  // permutation halves, padded to a multiple of 256 (padding repeats real ones)
    const uint32_t *b_lo7;      // b_lo + 7 (mod 2^32): the addend of the two-phase kernel's cheap value L'
    int k;                      // num_perm
    const void *init;           // running signatures to merge, or nullptr
    int64_t init_stride;        // elements between init rows (0 = broadcast one row)
    int init_is_u64;
    void *out;                  // [n_docs, k] u32 or u64
    int out_is_u64;
    unsigned *work_counter;     // [K slices] device counters, zeroed by the launcher: dynamic unit distribution
    int docs_per_unit;          // 0 = chosen by the launcher; > 0 = forced (tests)
    // fused all-gather epilogue: when n_peers > 0 every signature row is stored into each peer_out[p]
    // (the full [N_total, k] matrix of rank p, mapped peer memory) at row peer_row_offset + d
    int n_peers;
    int64_t peer_row_offset;
    void *peer_out[8];
    // long documents (signature_kernel.cu): a document longer than long_doc_tokens is not processed by the warp that
    // meets it; the warp stores the row's initial value and appends ceil(len / 2^piece_shift) PieceDesc entries, which a
    // second launch of the kernel in piece mode spreads over all warps and min-merges into the row with atomicMin.
    int64_t long_doc_tokens;    // 0 = never defer
    int piece_shift;            // log2 of the piece length in tokens
    unsigned *piece_hdr;        // [0] = pieces appended so far; [64 + K-slice] = work counters of the piece-mode launch
    struct PieceDesc *pieces;   // capacity guaranteed by the caller: n_tokens / 2^piece_shift + n_tokens / long_doc_tokens + 2
    // general variants of the signature kernel (appended last: the layout the default variant sees stays as it was)
    const uint32_t *b_lo8;      // b_lo + 8: the addend of L' when `% p` may take its conditional subtract (window 8)
    int gen;                    // 0 = u32 tokens + safe permutations, 1 = u32 tokens + any permutations, 2 = u64 tokens
    // fused LSH insert (signature_kernel.cu, template LSH): when lsh_slots != nullptr the warp that finishes document d also
    // inserts it into the device-resident LSH index as document lsh_doc0 + d (the bucket tables' DRAM latency hides behind the
    // other warps' integer work); `out` then is the index's own signature storage (u32, row lsh_doc0 + d at out + d * k)
    uint64_t *lsh_slots;        // LshDev::slots
    int32_t *lsh_next;          // LshDev::next
    int64_t lsh_cap_slots, lsh_doc0;
    int lsh_b, lsh_r;
};
struct PieceDesc { int64_t row, start, end, reserved; };
constexpr int kPieceHdrBytes = 512;
constexpr int64_t kLongDocTokensApi = 4096;   // documents longer than this are cut into pieces of 2^kPieceShiftApi tokens
constexpr int kPieceShiftApi = 10;
enum { MODE_TWO_PHASE = 0, MODE_DIRECT = 1, MODE_EXACT = 2 };
cudaError_t launch_minhash_bulk(const BulkParams &prm, int mode, int token_is_u64, int sm_count, cudaStream_t s);
cudaError_t launch_minhash_sig(const BulkParams &prm, int sm_count, cudaStream_t s);   // signature_kernel.cu (two-phase; variant = prm.gen)
size_t minhash_sig_workspace_bytes(int64_t n_tokens);   // piece table for long documents (0 if none can occur)
cudaError_t launch_seg_min(const uint32_t *part, const int64_t *seg, int64_t n_docs, int k, const void *init,
                           int64_t init_stride, int init_is_u64, void *out, int out_is_u64, int sm_count,
                           cudaStream_t s);
cudaError_t launch_sig_merge_min(const uint32_t *x, const uint32_t *y, int64_t n, uint32_t *out, int sm_count,
                                 cudaStream_t s);

cudaError_t launch_lean_pack(const void *sig, int sig_is_u64, int64_t n, int k, int64_t seed, int big_endian,
                             uint8_t *rec, int sm_count, cudaStream_t s);
cudaError_t launch_lean_unpack(const uint8_t *rec, int64_t n, int k, int64_t seed, int big_endian, void *sig,
                               int sig_is_u64, int *d_status, int sm_count, cudaStream_t s);
cudaError_t launch_band_keys_be(const uint32_t *sig, int64_t n, int k, int b, int r, uint8_t *out, int sm_count,
                                cudaStream_t s);
cudaError_t launch_band_fingerprints(const uint32_t *sig, int64_t n, int k, int b, int r, uint64_t *out, int sm_count,
                                     cudaStream_t s);

cudaError_t launch_band_sums(const uint32_t *sig, int64_t n, int k, int b, int r, uint64_t *keys, int sm_count, cudaStream_t s);
cudaError_t launch_bloom_insert(const uint32_t *sig, int64_t n, int k, int b, int r, uint32_t *bits, uint64_t words_per_table,
                                uint64_t n_bits, int n_hashes, int sm_count, cudaStream_t s);
cudaError_t launch_bloom_query(const uint32_t *sig, int64_t n, int k, int b, int r, const uint32_t *bits,
                               uint64_t words_per_table, uint64_t n_bits, int n_hashes, uint8_t *hit, int sm_count,
                               cudaStream_t s);

cudaError_t launch_wmh_transpose(const float *src, int ss, int dim, int ss_pad, float *dst, cudaStream_t s);
cudaError_t launch_wmh(const float *rs_t, const float *lncs_t, const float *betas_t, int ss, int ss_pad, int dim,
                       const float *v, int64_t n, int64_t *out, int32_t *status, int many, int input_log, int sm_count,
                       cudaStream_t s);

// ---- device-resident LSH index (lsh_kernels.cu) -------------------------------------------------
struct LshDev {
    uint32_t *sig;        // [cap_docs][k] copies of the inserted signatures (tuple verification)
    // [b][cap_slots] 16-byte slots {uint64 fingerprint, int32 head, int32 unused}: the claim (atomicCAS on the key) and the
    // chain update (atomicExch on the head = most recently inserted doc of the bucket, -1 = none) touch ONE 32-byte sector
    uint64_t *slots;
    int32_t *next;        // [cap_docs][b]   next doc in the same bucket of that band, -1 = end
    int64_t cap_docs, cap_slots;  // cap_slots is a power of two >= 2 * cap_docs
    int k, b, r;
};
cudaError_t launch_lsh_insert(const LshDev &ix, const uint32_t *new_sig, int64_t doc0, int64_t n_new, int sm_count,
                              cudaStream_t s);
cudaError_t launch_lsh_query(const LshDev &ix, const uint32_t *qsig, int64_t nq, int64_t n_docs, int64_t *counts,
                             const int64_t *ptr, int32_t *out, int fill, int sm_count, cudaStream_t s);
cudaError_t launch_exclusive_scan(const int64_t *in, int64_t n, int64_t *out, int64_t *scratch, cudaStream_t s);

cudaError_t launch_jaccard_pairs(const uint32_t *sig, int64_t n_rows, int k, const int64_t *ia, const int64_t *ib,
                                 int64_t m, int32_t *out, int sm_count, cudaStream_t s);

cudaError_t launch_jaccard_topk(const uint32_t *q, int64_t nq, const uint32_t *db, int64_t n, int k, int topk,
                                int64_t self_base, int32_t *out_cnt, int64_t *out_idx, int sm_count, cudaStream_t s);

size_t jaccard_topk_workspace_bytes(int64_t nq, int64_t n, int k);
cudaError_t launch_jaccard_topk_pf(const uint32_t *q, int64_t nq, const uint32_t *db, int64_t n, int k, int topk,
                                   int64_t self_base, int32_t *out_cnt, int64_t *out_idx, void *workspace, int sm_count,
                                   cudaStream_t s);

cudaError_t launch_sha1_tokens(const uint8_t *bytes, const int64_t *off, int64_t n_tok, void *out, int out_is_u64,
                               int sm_count, cudaStream_t s);
cudaError_t launch_hash_tokens(const uint8_t *bytes, const int64_t *off, int64_t n_tok, int kind, uint32_t seed,
                               uint32_t *out, int sm_count, cudaStream_t s);

cudaError_t launch_bbit_pack(const uint32_t *sig, int64_t n, int k, int b, int slot, uint64_t *out, int sm_count,
                             cudaStream_t s);
cudaError_t launch_bbit_unpack(const uint64_t *blocks, int64_t n, int k, int slot, uint32_t *sig, int sm_count,
                               cudaStream_t s);

cudaError_t launch_forest_query(const uint32_t *sig, const int32_t *order, int64_t n, int K, int l, int k,
                                const uint32_t *qsig, int64_t nq, int topk, int32_t *out, int sm_count,
                                cudaStream_t s);

// ---- PTX helpers -----------------------------------------------------------------
#ifndef DSK_EMU
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// make mbarrier.init visible to the async (TMA) proxy
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// 1-D bulk async copy global -> shared (TMA engine; SASS: UBLKCP).  dst/src 16-byte
// aligned, bytes a multiple of 16; completion is signalled as tx-bytes on `bar`.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// 1-D bulk async copy shared -> global (SASS: UBLKCP / UTMASTG family), bulk-group completion.
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ uint32_t umin3(uint32_t a, uint32_t b, uint32_t c) { return min(min(a, b), c); }
#endif  // !DSK_EMU

// ---- LSH bucket fingerprints (lsh_kernels.cu; the signature kernel's fused insert epilogue) ------------------------------
constexpr uint64_t kEmptyKey = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ uint64_t lsh_mix64(uint64_t h) {
    h ^= h >> 32; h *= 0xD6E8FEB86659FD93ull; h ^= h >> 32; h *= 0xD6E8FEB86659FD93ull; h ^= h >> 32;
    return h;
}

__device__ __forceinline__ uint64_t band_fp(const uint32_t *v, int r, int band) {
    uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t)band;
    for (int q = 0; q < r; ++q) h = (h ^ v[q]) * 0xFF51AFD7ED558CCDull + 0x2545F4914F6CDD1Dull;
    h = lsh_mix64(h);
    return h == kEmptyKey ? h - 1 : h;
}

}  // namespace dsk
