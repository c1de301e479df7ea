// jaccard_kernels.cu -- Jaccard estimate = count of equal signature positions / K
// (datasketch/minhash.py:324, inherited by LeanMinHash) on sm_100a.
//
//  jaccard_pairs : m explicit (i, j) pairs over a [N, K] u32 signature matrix.  HBM-bound gather:
//                  2 * 4K bytes in, 4 bytes out per pair.  warp <-> pair, lanes read the two rows
//                  with 128-bit loads, compare, popc-free add, warp-shuffle reduce.
//  jaccard_topk  : for each query row the `topk` database rows with the most equal positions
//                  (ties -> lower index, optional self-exclusion): tiled all-pairs compare with
//                  register blocking; see the kernel comment.
#include "dsk_common.cuh"

namespace dsk {

__device__ __forceinline__ int eq4(const uint4 a, const uint4 b) {
    return (a.x == b.x) + (a.y == b.y) + (a.z == b.z) + (a.w == b.w);
}

__global__ void __launch_bounds__(256) jaccard_pairs_kernel(const uint32_t *__restrict__ sig, int64_t n_rows, int k,
                                                            const int64_t *__restrict__ ia,
                                                            const int64_t *__restrict__ ib, int64_t m,
                                                            int32_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const bool vec = (k & 3) == 0;
    for (int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < m; p += warps) {
        const int64_t i = __ldg(ia + p), j = __ldg(ib + p);
        int cnt = 0;
        if (i >= 0 && i < n_rows && j >= 0 && j < n_rows) {
            const uint32_t *x = sig + i * k, *y = sig + j * k;
            if (vec) {
                const uint4 *x4 = reinterpret_cast<const uint4 *>(x), *y4 = reinterpret_cast<const uint4 *>(y);
                for (int c = lane; c < (k >> 2); c += 32) cnt += eq4(__ldg(x4 + c), __ldg(y4 + c));
            } else {
                for (int c = lane; c < k; c += 32) cnt += (__ldg(x + c) == __ldg(y + c));
            }
        } else {
            cnt = (lane == 0) ? -1 : 0;  // out-of-range pair index -> -1
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, o);
        if (lane == 0) out[p] = cnt;
    }
}

// ---- all-pairs top-k -----------------------------------------------------------------------------
// CTA tile: kTQ = 64 query rows x kTD = 128 database rows per step; 128 threads, thread <-> 8 queries x
// 8 database rows (64 counters in registers).  Both tiles are staged TRANSPOSED in shared memory
// ([position][row]) so a thread reads its 8 + 8 values of one signature position with four LDS.128.
// The query tile is staged whole, once per query tile, when it fits a block's 227 KB of shared memory
// (K <= 736); above that (WHOLE_Q = false) it goes through shared memory kKc positions at a time next to
// the database chunk, a footprint of 49 KB whatever K, so every num_perm the API accepts runs.
// After a database tile, counts above the query's current k-th best are inserted into the query's
// sorted list in shared memory (ties keep the lower database index because tiles arrive in index
// order and insertion requires a strictly larger count than the k-th entry ... or an unfilled slot).
constexpr int kTQ = 64, kTD = 128, kKc = 32, kTopThreads = 128, kMaxTopK = 32;

struct TopkParams {
    const uint32_t *q;    // [nq, k]
    const uint32_t *db;   // [n, k]
    int64_t nq, n;
    int k, topk;
    int64_t self_base;    // query i is database row self_base + i (excluded), or < 0
    int32_t *out_cnt;     // [nq, topk]
    int64_t *out_idx;     // [nq, topk]  (-1 = no such row)
};

template <bool WHOLE_Q>
__global__ void __launch_bounds__(kTopThreads) jaccard_topk_kernel(const TopkParams p) {
    DSK_DYNAMIC_SMEM_T(uint32_t, sm, 16);
    const int K = p.k;
    const int kpad = (K + kKc - 1) / kKc * kKc;
    uint32_t *sQ = sm;                                              // [kpad][kTQ] (WHOLE_Q) or [kKc][kTQ]
    uint32_t *sD = sQ + (size_t)(WHOLE_Q ? kpad : kKc) * kTQ;      // [kKc][kTD]
    int32_t *top_cnt = reinterpret_cast<int32_t *>(sD + kKc * kTD);   // [kTQ][topk]
    int64_t *top_idx = reinterpret_cast<int64_t *>(top_cnt + kTQ * kMaxTopK);  // [kTQ][topk]
    int *lock = reinterpret_cast<int *>(top_idx + kTQ * kMaxTopK);    // [kTQ]
    volatile int32_t *thr = reinterpret_cast<volatile int32_t *>(lock + kTQ);  // [kTQ] k-th best count, -1 while unfilled
    volatile int64_t *kidx = reinterpret_cast<volatile int64_t *>(const_cast<int32_t *>(thr) + kTQ);  // [kTQ] its index

    const int tid = threadIdx.x;
    const int qg = tid >> 4, dg = tid & 15;         // 8 query groups x 16 database groups
    const int topk = p.topk;
    const bool qvec = (K & 3) == 0 && (reinterpret_cast<uintptr_t>(p.q) & 15) == 0;   // the API checks only d_db's alignment

    for (int64_t qt = blockIdx.x; qt * kTQ < p.nq; qt += gridDim.x) {
        const int64_t q0 = qt * kTQ;
        __syncthreads();
        for (int i = tid; i < kTQ * kMaxTopK; i += kTopThreads) { top_cnt[i] = -1; top_idx[i] = -1; }
        for (int i = tid; i < kTQ; i += kTopThreads) { lock[i] = 0; thr[i] = -1; kidx[i] = -1; }
        if (WHOLE_Q) {
            // query tile, transposed; rows / positions beyond the data are filled so they never match
            for (int e = tid; e < kTQ * kpad; e += kTopThreads) {
                const int r = e / kpad, c = e - r * kpad;
                uint32_t v = 0x51EDu + (uint32_t)c;           // padded positions never match: the db side uses ~filler
                if (q0 + r < p.nq && c < K) v = __ldg(p.q + (q0 + r) * (int64_t)K + c);
                sQ[(size_t)c * kTQ + r] = v;
            }
            __syncthreads();
        }

        for (int64_t d0 = 0; d0 < p.n; d0 += kTD) {
            int cnt[8][8];
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) cnt[a][b] = 0;
            for (int c0 = 0; c0 < kpad; c0 += kKc) {
                __syncthreads();
                // stage query chunk [kTQ rows][kKc positions] transposed: each task = (row, 8 positions); rows and
                // positions beyond the data get a filler that the database side never holds at that position
                for (int task = tid; !WHOLE_Q && task < kTQ * (kKc / 8); task += kTopThreads) {
                    const int r = task % kTQ, seg = task / kTQ;
                    const int64_t row = q0 + r;
                    const int cb = c0 + seg * 8;
                    uint32_t v[8];
                    if (row < p.nq && qvec && cb + 8 <= K) {
                        const uint4 x = __ldg(reinterpret_cast<const uint4 *>(p.q + row * (int64_t)K + cb));
                        const uint4 y = __ldg(reinterpret_cast<const uint4 *>(p.q + row * (int64_t)K + cb + 4));
                        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
                    } else {
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            v[u] = 0x51EDu + (uint32_t)(cb + u);
                            if (row < p.nq && cb + u < K) v[u] = __ldg(p.q + row * (int64_t)K + cb + u);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) sQ[(seg * 8 + u) * kTQ + r] = v[u];
                }
                // stage database chunk [kTD rows][kKc positions] transposed: each task = (row, 8 positions)
                for (int task = tid; task < kTD * (kKc / 8); task += kTopThreads) {
                    const int r = task % kTD, seg = task / kTD;
                    const int64_t row = d0 + r;
                    const int cb = c0 + seg * 8;
                    uint32_t v[8];
                    if (row < p.n && (K & 3) == 0 && cb + 8 <= K) {   // one full 32-byte sector per task
                        const uint4 x = __ldg(reinterpret_cast<const uint4 *>(p.db + row * (int64_t)K + cb));
                        const uint4 y = __ldg(reinterpret_cast<const uint4 *>(p.db + row * (int64_t)K + cb + 4));
                        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
                    } else {
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            v[u] = ~(0x51EDu + (uint32_t)(cb + u));  // never equals the query filler at this position
                            if (row < p.n && cb + u < K) v[u] = __ldg(p.db + row * (int64_t)K + cb + u);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) sD[(seg * 8 + u) * kTD + r] = v[u];
                }
                __syncthreads();
#pragma unroll 4
                for (int cc = 0; cc < kKc; ++cc) {
                    const uint32_t *qrow = sQ + (size_t)((WHOLE_Q ? c0 : 0) + cc) * kTQ;
                    const uint4 qa = *reinterpret_cast<const uint4 *>(qrow + qg * 8);
                    const uint4 qb = *reinterpret_cast<const uint4 *>(qrow + qg * 8 + 4);
                    const uint4 da = *reinterpret_cast<const uint4 *>(sD + cc * kTD + dg * 8);
                    const uint4 db = *reinterpret_cast<const uint4 *>(sD + cc * kTD + dg * 8 + 4);
                    const uint32_t qv[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
                    const uint32_t dv[8] = {da.x, da.y, da.z, da.w, db.x, db.y, db.z, db.w};
#pragma unroll
                    for (int a = 0; a < 8; ++a)
#pragma unroll
                        for (int b = 0; b < 8; ++b) cnt[a][b] += (qv[a] == dv[b]);
                }
            }
            // fold this tile's counts into the per-query sorted lists
#pragma unroll
            for (int a = 0; a < 8; ++a) {
                const int ql = qg * 8 + a;
                const int64_t qrow = q0 + ql;
                if (qrow >= p.nq) continue;
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    const int64_t drow = d0 + dg * 8 + b;
                    if (drow >= p.n) continue;
                    if (p.self_base >= 0 && drow == p.self_base + qrow) continue;
                    const int c = cnt[a][b];
                    {   // cheap filter (re-checked under the lock): worse than the current k-th entry?
                        const int32_t t = thr[ql];
                        if (c < t || (c == t && drow > kidx[ql])) continue;
                    }
                    bool done = false;
                    while (!done) {
                        if (atomicCAS(&lock[ql], 0, 1) == 0) {
                            int32_t *tc = top_cnt + ql * kMaxTopK;
                            int64_t *ti = top_idx + ql * kMaxTopK;
                            // position: after every entry with count > c, or count == c and lower index
                            int pos = topk;
                            for (int s = 0; s < topk; ++s) {
                                const int32_t sc = tc[s];
                                if (sc < c || (sc == c && (ti[s] < 0 || ti[s] > drow))) { pos = s; break; }
                            }
                            if (pos < topk) {
                                for (int s = topk - 1; s > pos; --s) { tc[s] = tc[s - 1]; ti[s] = ti[s - 1]; }
                                tc[pos] = c; ti[pos] = drow;
                                kidx[ql] = ti[topk - 1];
                                thr[ql] = (ti[topk - 1] < 0) ? -1 : tc[topk - 1];
                            }
                            __threadfence_block();
                            atomicExch(&lock[ql], 0);
                            done = true;
                        }
                    }
                }
            }
        }
        __syncthreads();
        for (int e = tid; e < kTQ * topk; e += kTopThreads) {
            const int r = e / topk, s = e - r * topk;
            if (q0 + r < p.nq) {
                p.out_cnt[(q0 + r) * topk + s] = top_cnt[r * kMaxTopK + s];
                p.out_idx[(q0 + r) * topk + s] = top_idx[r * kMaxTopK + s];
            }
        }
    }
}

// ---- all-pairs top-k with a bit-sliced fingerprint prefilter --------------------------------------------------
// The exact kernel above spends 2 ALU ops per (pair, position).  Here every signature value is first reduced to a
// 16-bit fingerprint stored BIT-SLICED: plane p, word w of a row holds bit p of the fingerprints of positions
// 32w .. 32w+31.  For a pair, AND_p ~(Q_p ^ D_p) has a 1 exactly where all 16 fingerprint bits agree, so
//     ub = sum_w popc(AND_p ~(Q_p[w] ^ D_p[w]))  >=  number of equal positions          (equal values agree in every bit)
// costs 16 LOP3 + POPC + IADD per 32 positions = 0.56 op per position, and for unrelated values exceeds the true count
// by K / 65536 on average.  A pair goes on to the exact count (and the sorted list) only if its upper bound could still
// enter the query's top-k; since ub >= count no pair that belongs in the list is ever dropped -- results are identical to
// the exact kernel (MinHash.jaccard, minhash.py:324).  Plane layout (written by fp_planes_kernel): [tile][plane][word][row
// in tile], so a tile is one contiguous block whose (plane, word) lines are read with LDS.128 over rows.
constexpr int kPfB = 16;

__global__ void __launch_bounds__(256) fp_planes_kernel(const uint32_t *__restrict__ sig, int64_t n, int k, int words,
                                                        int rows_per_tile, int pad_bit, uint32_t *__restrict__ planes) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t n_pad = (n + rows_per_tile - 1) / rows_per_tile * rows_per_tile;
    const int64_t items = n_pad * words;
    for (int64_t it = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); it < items; it += warps) {
        const int64_t row = it / words;
        const int w = (int)(it - row * words);
        const int c = w * 32 + lane;
        uint32_t f = 0;
        bool pad = true;
        if (row < n && c < k) {
            const uint32_t v = __ldg(sig + row * (int64_t)k + c);
            f = (v ^ (v >> 16)) & 0xFFFFu;
            pad = false;
        }
        const int64_t tile = row / rows_per_tile;
        const int r = (int)(row - tile * rows_per_tile);
        uint32_t *base = planes + (tile * kPfB * words + w) * rows_per_tile + r;
#pragma unroll
        for (int pl = 0; pl < kPfB; ++pl) {
            // positions beyond K (and rows beyond n): plane 0 differs between the two sides, so they never agree
            const bool bit = pad ? (pl == 0 && pad_bit) : ((f >> pl) & 1u);
            const unsigned word = __ballot_sync(0xFFFFFFFFu, bit);
            if (lane == 0) base[(int64_t)pl * words * rows_per_tile] = word;
        }
    }
}

struct TopkPfParams {
    const uint32_t *q, *db;        // [nq, k], [n, k]  (exact counts of the surviving pairs)
    const uint32_t *qpl, *dpl;     // bit planes, [tile][16][words][kTQ] / [tile][16][words][kTD]
    int64_t nq, n;
    int k, words, topk;
    int64_t self_base;
    int32_t *out_cnt;
    int64_t *out_idx;
};

__global__ void __launch_bounds__(kTopThreads) jaccard_topk_pf_kernel(const TopkPfParams p) {
    DSK_DYNAMIC_SMEM_T(uint32_t, sm, 16);
    const int W = p.words;
    uint32_t *sQ = sm;                                   // [16][W][kTQ]
    uint32_t *sD = sQ + (size_t)kPfB * W * kTQ;          // [16][W][kTD]
    int32_t *top_cnt = reinterpret_cast<int32_t *>(sD + (size_t)kPfB * W * kTD);   // [kTQ][kMaxTopK]
    int64_t *top_idx = reinterpret_cast<int64_t *>(top_cnt + kTQ * kMaxTopK);
    int *lock = reinterpret_cast<int *>(top_idx + kTQ * kMaxTopK);                 // [kTQ]
    volatile int32_t *thr = reinterpret_cast<volatile int32_t *>(lock + kTQ);      // [kTQ] k-th best count, -1 while unfilled
    volatile int64_t *kidx = reinterpret_cast<volatile int64_t *>(const_cast<int32_t *>(thr) + kTQ);   // [kTQ]
    unsigned *qn = reinterpret_cast<unsigned *>(const_cast<int64_t *>(kidx) + kTQ);                    // candidate count
    uint16_t *queue = reinterpret_cast<uint16_t *>(qn + 4);                                            // [kTQ * kTD]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int qg = tid >> 4, dg = tid & 15;         // 8 query groups x 16 database groups
    const int topk = p.topk, K = p.k;
    const size_t qtile_words = (size_t)kPfB * W * kTQ, dtile_words = (size_t)kPfB * W * kTD;

    for (int64_t qt = blockIdx.x; qt * kTQ < p.nq; qt += gridDim.x) {
        const int64_t q0 = qt * kTQ;
        __syncthreads();
        for (int i = tid; i < kTQ * kMaxTopK; i += kTopThreads) { top_cnt[i] = -1; top_idx[i] = -1; }
        for (int i = tid; i < kTQ; i += kTopThreads) { lock[i] = 0; thr[i] = -1; kidx[i] = -1; }
        if (tid == 0) *qn = 0;
        {
            const uint4 *src = reinterpret_cast<const uint4 *>(p.qpl + qt * qtile_words);
            for (size_t e = tid; e < qtile_words / 4; e += kTopThreads) reinterpret_cast<uint4 *>(sQ)[e] = __ldg(src + e);
        }
        for (int64_t d0 = 0; d0 < p.n; d0 += kTD) {
            __syncthreads();
            {
                const uint4 *src = reinterpret_cast<const uint4 *>(p.dpl + (d0 / kTD) * dtile_words);
                for (size_t e = tid; e < dtile_words / 4; e += kTopThreads) reinterpret_cast<uint4 *>(sD)[e] = __ldg(src + e);
            }
            __syncthreads();
            int cnt[8][8];
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) cnt[a][b] = 0;
            for (int w = 0; w < W; ++w) {
                uint32_t t[8][8];
#pragma unroll
                for (int pl = 0; pl < kPfB; ++pl) {
                    const uint32_t *ql = sQ + ((size_t)pl * W + w) * kTQ + qg * 8;
                    const uint32_t *dl = sD + ((size_t)pl * W + w) * kTD + dg * 8;
                    const uint4 qa = *reinterpret_cast<const uint4 *>(ql), qb = *reinterpret_cast<const uint4 *>(ql + 4);
                    const uint4 da = *reinterpret_cast<const uint4 *>(dl), db = *reinterpret_cast<const uint4 *>(dl + 4);
                    const uint32_t qv[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
                    const uint32_t dv[8] = {da.x, da.y, da.z, da.w, db.x, db.y, db.z, db.w};
#pragma unroll
                    for (int a = 0; a < 8; ++a)
#pragma unroll
                        for (int b = 0; b < 8; ++b) {
                            const uint32_t same = ~(qv[a] ^ dv[b]);
                            t[a][b] = pl == 0 ? same : (t[a][b] & same);          // one LOP3
                        }
                }
#pragma unroll
                for (int a = 0; a < 8; ++a)
#pragma unroll
                    for (int b = 0; b < 8; ++b) cnt[a][b] += __popc(t[a][b]);
            }
            // pairs whose upper bound could still enter the query's list go on to the exact count
#pragma unroll
            for (int a = 0; a < 8; ++a) {
                const int ql = qg * 8 + a;
                const int64_t qrow = q0 + ql;
                if (qrow >= p.nq) continue;
                const int32_t tq = thr[ql];
                const int64_t kq = kidx[ql];
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    const int dl = dg * 8 + b;
                    const int64_t drow = d0 + dl;
                    if (drow >= p.n) continue;
                    if (p.self_base >= 0 && drow == p.self_base + qrow) continue;
                    const int ub = cnt[a][b];
                    if (ub < tq || (ub == tq && drow > kq)) continue;
                    queue[atomicAdd(qn, 1u)] = (uint16_t)((ql << 7) | dl);
                }
            }
            __syncthreads();
            const unsigned nc = *qn;
            for (unsigned ci = warp; ci < nc; ci += kTopThreads / 32) {
                const unsigned ent = queue[ci];
                const int ql = (int)(ent >> 7), dl = (int)(ent & 127u);
                const int64_t qrow = q0 + ql, drow = d0 + dl;
                const uint32_t *x = p.q + qrow * (int64_t)K, *y = p.db + drow * (int64_t)K;
                int c = 0;
                for (int e = lane; e < K; e += 32) c += (__ldg(x + e) == __ldg(y + e));
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
                if (lane == 0) {
                    const int32_t tq = thr[ql];
                    if (!(c < tq || (c == tq && drow > kidx[ql]))) {
                        bool done = false;
                        while (!done) {
                            if (atomicCAS(&lock[ql], 0, 1) == 0) {
                                int32_t *tc = top_cnt + ql * kMaxTopK;
                                int64_t *ti = top_idx + ql * kMaxTopK;
                                int pos = topk;   // after every entry with count > c, or count == c and lower index
                                for (int s = 0; s < topk; ++s) {
                                    const int32_t sc = tc[s];
                                    if (sc < c || (sc == c && (ti[s] < 0 || ti[s] > drow))) { pos = s; break; }
                                }
                                if (pos < topk) {
                                    for (int s = topk - 1; s > pos; --s) { tc[s] = tc[s - 1]; ti[s] = ti[s - 1]; }
                                    tc[pos] = c; ti[pos] = drow;
                                    kidx[ql] = ti[topk - 1];
                                    thr[ql] = (ti[topk - 1] < 0) ? -1 : tc[topk - 1];
                                }
                                __threadfence_block();
                                atomicExch(&lock[ql], 0);
                                done = true;
                            }
                        }
                    }
                }
            }
            __syncthreads();
            if (tid == 0) *qn = 0;
        }
        __syncthreads();
        for (int e = tid; e < kTQ * topk; e += kTopThreads) {
            const int r = e / topk, s2 = e - r * topk;
            if (q0 + r < p.nq) {
                p.out_cnt[(q0 + r) * topk + s2] = top_cnt[r * kMaxTopK + s2];
                p.out_idx[(q0 + r) * topk + s2] = top_idx[r * kMaxTopK + s2];
            }
        }
    }
}

// dynamic shared memory of jaccard_topk_pf_kernel: both tiles' bit planes, the per-query lists and the candidate queue
size_t jaccard_topk_pf_smem(int k) {
    const int words = (k + 31) / 32;
    return (size_t)kPfB * words * (kTQ + kTD) * 4 + (size_t)kTQ * kMaxTopK * (4 + 8) + (size_t)kTQ * 16 + 16 +
           (size_t)kTQ * kTD * 2;
}

// the prefilter needs K >= 32 to pay off and its planes must fit a block's shared memory (K <= 480)
static bool jaccard_topk_pf_applies(int k) { return k >= 32 && jaccard_topk_pf_smem(k) <= kMaxDynamicSmemPerBlock; }

// workspace of the prefilter path: the bit planes of both matrices (0 = the path does not apply)
size_t jaccard_topk_workspace_bytes(int64_t nq, int64_t n, int k) {
    if (!jaccard_topk_pf_applies(k) || n < 4 * kTD) return 0;
    const int words = (k + 31) / 32;
    const size_t qt = (size_t)((nq + kTQ - 1) / kTQ), dt = (size_t)((n + kTD - 1) / kTD);
    return (qt * kTQ + dt * kTD) * (size_t)kPfB * words * sizeof(uint32_t);
}

// K whose planes do not fit (K > 480) runs the exact kernel instead; the workspace is then not touched
cudaError_t launch_jaccard_topk_pf(const uint32_t *q, int64_t nq, const uint32_t *db, int64_t n, int k, int topk,
                                   int64_t self_base, int32_t *out_cnt, int64_t *out_idx, void *workspace, int sm_count,
                                   cudaStream_t s) {
    if (nq <= 0) return cudaSuccess;
    if (jaccard_topk_pf_smem(k) > kMaxDynamicSmemPerBlock)
        return launch_jaccard_topk(q, nq, db, n, k, topk, self_base, out_cnt, out_idx, sm_count, s);
    const int words = (k + 31) / 32;
    const size_t qt = (size_t)((nq + kTQ - 1) / kTQ);
    uint32_t *qpl = static_cast<uint32_t *>(workspace);
    uint32_t *dpl = qpl + qt * kTQ * (size_t)kPfB * words;
    const int pgrid = sm_count * 8;
    DSK_LAUNCH(fp_planes_kernel, pgrid, 256, 0, s, q, nq, k, words, kTQ, 0, qpl);
    DSK_LAUNCH(fp_planes_kernel, pgrid, 256, 0, s, db, n, k, words, kTD, 1, dpl);
    TopkPfParams p;
    p.q = q; p.db = db; p.qpl = qpl; p.dpl = dpl; p.nq = nq; p.n = n; p.k = k; p.words = words; p.topk = topk;
    p.self_base = self_base; p.out_cnt = out_cnt; p.out_idx = out_idx;
    const size_t smem = jaccard_topk_pf_smem(k);
    cudaError_t e = cudaFuncSetAttribute(jaccard_topk_pf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int64_t grid = (nq + kTQ - 1) / kTQ;
    if (grid > (int64_t)sm_count * 2) grid = (int64_t)sm_count * 2;
    DSK_LAUNCH(jaccard_topk_pf_kernel, (unsigned)grid, kTopThreads, smem, s, p);
    return cudaGetLastError();
}

// dynamic shared memory of jaccard_topk_kernel: the query tile (whole, or one kKc chunk), the database chunk, the lists
size_t jaccard_topk_smem(int k, bool whole_q) {
    const int kpad = (k + kKc - 1) / kKc * kKc;
    return (size_t)(whole_q ? kpad : kKc) * kTQ * 4 + (size_t)kKc * kTD * 4 + (size_t)kTQ * kMaxTopK * (4 + 8) +
           (size_t)kTQ * 16;
}

cudaError_t launch_jaccard_topk(const uint32_t *q, int64_t nq, const uint32_t *db, int64_t n, int k, int topk,
                                int64_t self_base, int32_t *out_cnt, int64_t *out_idx, int sm_count, cudaStream_t s) {
    if (nq <= 0) return cudaSuccess;
    TopkParams p;
    p.q = q; p.db = db; p.nq = nq; p.n = n; p.k = k; p.topk = topk; p.self_base = self_base;
    p.out_cnt = out_cnt; p.out_idx = out_idx;
    const bool whole_q = jaccard_topk_smem(k, true) <= kMaxDynamicSmemPerBlock;
    const size_t smem = jaccard_topk_smem(k, whole_q);
    cudaError_t e = whole_q
        ? cudaFuncSetAttribute(jaccard_topk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
        : cudaFuncSetAttribute(jaccard_topk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int64_t grid = (nq + kTQ - 1) / kTQ;
    if (grid > (int64_t)sm_count * 3) grid = (int64_t)sm_count * 3;
    if (whole_q) DSK_LAUNCH((jaccard_topk_kernel<true>), (unsigned)grid, kTopThreads, smem, s, p);
    else DSK_LAUNCH((jaccard_topk_kernel<false>), (unsigned)grid, kTopThreads, smem, s, p);
    return cudaGetLastError();
}

cudaError_t launch_jaccard_pairs(const uint32_t *sig, int64_t n_rows, int k, const int64_t *ia, const int64_t *ib,
                                 int64_t m, int32_t *out, int sm_count, cudaStream_t s) {
    if (m <= 0) return cudaSuccess;
    int64_t grid = (m + 7) / 8;
    if (grid > (int64_t)sm_count * 8) grid = (int64_t)sm_count * 8;
    DSK_LAUNCH(jaccard_pairs_kernel, (unsigned)grid, 256, 0, s, sig, n_rows, k, ia, ib, m, out);
    return cudaGetLastError();
}

}  // namespace dsk
