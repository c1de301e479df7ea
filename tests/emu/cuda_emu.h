// cuda_emu.h -- TEST INFRASTRUCTURE ONLY.  A minimal SIMT shim that lets g++ compile the *unmodified* kernel
// source of datasketch_b200/csrc/minhash_kernels.cu (with -DDSK_EMU) and run it on the CPU: every CUDA thread is
// a host thread, a warp's collectives (__syncwarp, __shfl_sync, __all_sync, __any_sync) are pthread barriers over its
// 32 lanes, __shared__ becomes static storage (CTAs run one after the other), and the mbarrier / bulk-copy PTX helpers
// are replaced by a phase counter + memcpy.  It exists so that the kernel's control logic (ring protocol, block
// patching, two-phase tracking, re-scan rules) is exercised against the oracle in the CPU test-suite, and so that
// ThreadSanitizer can check the shared-memory ring for missing synchronisation.  It says nothing about performance.
#pragma once
#include <pthread.h>
#include <sched.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <math.h>

#include <atomic>
#include <map>
#include <mutex>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __shared__ static
#define __align__(n) __attribute__((aligned(n)))

typedef int cudaError_t;
typedef void *cudaStream_t;
enum { cudaSuccess = 0 };
enum { cudaErrorInvalidValue = 1, cudaErrorMemoryAllocation = 2, cudaErrorInsufficientDriver = 35, cudaErrorNoDevice = 100 };
enum { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };

// ---- shared-memory limits of an sm_100 block, enforced like the driver does: a launch may use 48 KB of dynamic shared
// memory, or up to what cudaFuncSetAttribute raised the kernel's limit to, and that may not exceed 227 KB.  A launch
// over its limit runs nothing and leaves the error for cudaGetLastError.
constexpr size_t kEmuSmemDefault = 48 << 10, kEmuSmemOptin = 232448;
static inline cudaError_t &emu_last_error() { static thread_local cudaError_t e = cudaSuccess; return e; }
static inline cudaError_t cudaGetLastError() {
    const cudaError_t e = emu_last_error();
    emu_last_error() = cudaSuccess;
    return e;
}
static inline std::map<const void *, size_t> &emu_smem_limits() { static std::map<const void *, size_t> m; return m; }
static inline std::mutex &emu_smem_mu() { static std::mutex m; return m; }
template <typename F>
static inline cudaError_t cudaFuncSetAttribute(F kernel, int attr, int value) {
    if (attr != cudaFuncAttributeMaxDynamicSharedMemorySize) return cudaSuccess;
    if (value < 0 || (size_t)value > kEmuSmemOptin) return cudaErrorInvalidValue;
    std::lock_guard<std::mutex> lk(emu_smem_mu());
    emu_smem_limits()[reinterpret_cast<const void *>(kernel)] = (size_t)value;
    return cudaSuccess;
}
static inline size_t emu_smem_limit(const void *kernel) {
    std::lock_guard<std::mutex> lk(emu_smem_mu());
    const auto it = emu_smem_limits().find(kernel);
    return it == emu_smem_limits().end() ? kEmuSmemDefault : it->second;
}
static inline cudaError_t cudaMemsetAsync(void *p, int v, size_t n, cudaStream_t) { memset(p, v, n); return cudaSuccess; }

struct uint3e { unsigned x, y, z; };
struct uint2 { uint32_t x, y; };
struct uint4 { uint32_t x, y, z, w; };
struct float4 { float x, y, z, w; };
static inline uint2 make_uint2(uint32_t x, uint32_t y) { return uint2{x, y}; }
struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct ulonglong2 { unsigned long long x, y; };
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { return uint4{x, y, z, w}; }

extern thread_local uint3e threadIdx;
extern thread_local uint3e blockIdx;
extern thread_local uint3e gridDim;
extern thread_local uint3e blockDim;

// ---- integer min / max as CUDA declares them ------------------------------------------------------------------
#define DSK_EMU_MINMAX(T)                                      \
    static inline T min(T a, T b) { return b < a ? b : a; }    \
    static inline T max(T a, T b) { return a < b ? b : a; }
DSK_EMU_MINMAX(int)
DSK_EMU_MINMAX(unsigned)
DSK_EMU_MINMAX(long)
DSK_EMU_MINMAX(unsigned long)
DSK_EMU_MINMAX(long long)
DSK_EMU_MINMAX(unsigned long long)
#undef DSK_EMU_MINMAX

template <typename T>
static inline T __ldg(const T *p) { return *p; }

static inline unsigned atomicAdd(unsigned *p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }

// atomics: acquire-release so that ThreadSanitizer sees the lock / publish protocols the kernels build from them
static inline unsigned long long atomicCAS(unsigned long long *p, unsigned long long cmp, unsigned long long val) {
    __atomic_compare_exchange_n(p, &cmp, val, false, __ATOMIC_ACQ_REL, __ATOMIC_ACQUIRE);
    return cmp;
}
static inline unsigned atomicCAS(unsigned *p, unsigned cmp, unsigned val) {
    __atomic_compare_exchange_n(p, &cmp, val, false, __ATOMIC_ACQ_REL, __ATOMIC_ACQUIRE);
    return cmp;
}
static inline int atomicCAS(int *p, int cmp, int val) {
    const int want = cmp;
    __atomic_compare_exchange_n(p, &cmp, val, false, __ATOMIC_ACQ_REL, __ATOMIC_ACQUIRE);
    if (cmp != want) sched_yield();   // a failed claim is a spin on a lock another host thread holds: let it run
    return cmp;
}
static inline unsigned atomicMin(unsigned *p, unsigned v) {
    unsigned old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v < old && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_ACQ_REL, __ATOMIC_RELAXED)) {}
    return old;
}
static inline unsigned long long atomicMin(unsigned long long *p, unsigned long long v) {
    unsigned long long old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v < old && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_ACQ_REL, __ATOMIC_RELAXED)) {}
    return old;
}
static inline unsigned atomicOr(unsigned *p, unsigned v) { return __atomic_fetch_or(p, v, __ATOMIC_ACQ_REL); }
static inline unsigned atomicExch(unsigned *p, unsigned val) { return __atomic_exchange_n(p, val, __ATOMIC_ACQ_REL); }
static inline int atomicExch(int *p, int val) { return __atomic_exchange_n(p, val, __ATOMIC_ACQ_REL); }
static inline unsigned long long atomicExch(unsigned long long *p, unsigned long long val) { return __atomic_exchange_n(p, val, __ATOMIC_ACQ_REL); }
static inline void __threadfence_block() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }

// ---- CUDA runtime, synchronous and on host memory: "device" pointers are host pointers, one fake device with two SMs
enum { cudaStreamNonBlocking = 1 };
struct cudaDeviceProp { int multiProcessorCount, major, minor; size_t totalGlobalMem, sharedMemPerBlockOptin; char name[64]; };
static inline const char *cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : "emulated CUDA error"; }
static inline cudaError_t cudaGetDeviceCount(int *n) { *n = 1; return cudaSuccess; }
static inline cudaError_t cudaGetDevice(int *d) { *d = 0; return cudaSuccess; }
static inline cudaError_t cudaSetDevice(int d) { return d == 0 ? cudaSuccess : cudaErrorNoDevice; }
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp *p, int) {
    memset(p, 0, sizeof(*p));
    p->multiProcessorCount = 2; p->major = 10; p->minor = 0; p->totalGlobalMem = (size_t)8 << 30;
    p->sharedMemPerBlockOptin = kEmuSmemOptin;
    strcpy(p->name, "emulated sm_100 (host threads)");
    return cudaSuccess;
}
template <typename T>
static inline cudaError_t cudaMalloc(T **p, size_t n) {
    *p = static_cast<T *>(aligned_alloc(256, (n + 255) / 256 * 256 + 256));
    return *p ? cudaSuccess : cudaErrorMemoryAllocation;
}
template <typename T>
static inline cudaError_t cudaMallocHost(T **p, size_t n) { return cudaMalloc(p, n); }
static inline cudaError_t cudaFree(void *p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaFreeHost(void *p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaMemset(void *p, int v, size_t n) { memset(p, v, n); return cudaSuccess; }
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t *s, unsigned) { *s = nullptr; return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return cudaSuccess; }
typedef void *cudaEvent_t;   // streams are synchronous here: events are always "complete"
enum { cudaEventDisableTiming = 2 };
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t *e, unsigned) { *e = reinterpret_cast<void *>(1); return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return cudaSuccess; }

enum cudaMemcpyKind { cudaMemcpyHostToHost = 0, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice };
static inline cudaError_t cudaMemcpyAsync(void *dst, const void *src, size_t n, cudaMemcpyKind, cudaStream_t) {
    memcpy(dst, src, n);
    return cudaSuccess;
}
static inline cudaError_t cudaMemcpy(void *dst, const void *src, size_t n, cudaMemcpyKind) {
    memcpy(dst, src, n);
    return cudaSuccess;
}

// float32 operations rounded one by one (build the emulation with -ffp-contract=off so none are fused)
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline float __int_as_float(int v) { float f; memcpy(&f, &v, 4); return f; }
static inline uint32_t __funnelshift_l(uint32_t lo, uint32_t hi, int n) {
    n &= 31;
    return n ? (hi << n) | (lo >> (32 - n)) : hi;
}

// __byte_perm(x, y, s): byte i of the result = byte (s >> 4i) & 7 of the 8-byte value {y, x}
static inline uint32_t __byte_perm(uint32_t x, uint32_t y, uint32_t s) {
    const uint64_t v = ((uint64_t)y << 32) | x;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r |= (uint32_t)((v >> (8 * ((s >> (4 * i)) & 7))) & 0xFF) << (8 * i);
    return r;
}

// ---- one warp = 32 host threads ----------------------------------------------------------------------------------
struct EmuWarp {
    pthread_barrier_t bar;
    uint64_t slot[32];
    std::atomic<unsigned> votes_all, votes_any;
};
extern thread_local EmuWarp *emu_warp;
extern thread_local int emu_lane;

// one CTA = its warps + a CTA-wide barrier + the dynamic shared memory of the launch
struct EmuCta {
    pthread_barrier_t bar;
    unsigned char *dyn_smem;
};
extern thread_local EmuCta *emu_cta;
static inline void __syncthreads() { pthread_barrier_wait(&emu_cta->bar); }
static inline unsigned char *emu_dynamic_smem() { return emu_cta->dyn_smem; }

static inline void __syncwarp(unsigned = 0xFFFFFFFFu) { pthread_barrier_wait(&emu_warp->bar); }

template <typename T>
static inline T __shfl_sync(unsigned, T v, int src) {
    static_assert(sizeof(T) <= 8, "shuffle payload");
    uint64_t raw = 0;
    memcpy(&raw, &v, sizeof(T));
    emu_warp->slot[emu_lane] = raw;
    pthread_barrier_wait(&emu_warp->bar);
    raw = emu_warp->slot[src & 31];
    pthread_barrier_wait(&emu_warp->bar);
    T out;
    memcpy(&out, &raw, sizeof(T));
    return out;
}

template <typename T>
static inline T __shfl_xor_sync(unsigned m, T v, int mask) { return __shfl_sync(m, v, emu_lane ^ mask); }
template <typename T>
static inline T __shfl_up_sync(unsigned m, T v, int delta) {
    return __shfl_sync(m, v, emu_lane >= delta ? emu_lane - delta : emu_lane);
}

static inline unsigned emu_ballot(bool pred) {
    emu_warp->slot[emu_lane] = pred ? 1u : 0u;
    pthread_barrier_wait(&emu_warp->bar);
    unsigned m = 0;
    for (int i = 0; i < 32; ++i) m |= (unsigned)emu_warp->slot[i] << i;
    pthread_barrier_wait(&emu_warp->bar);
    return m;
}
static inline unsigned __ballot_sync(unsigned, int pred) { return emu_ballot(pred != 0); }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __ffs(unsigned v) { return __builtin_ffs((int)v); }
static inline unsigned __reduce_min_sync(unsigned, unsigned v) {   // redux.sync.min.u32
    emu_warp->slot[emu_lane] = v;
    pthread_barrier_wait(&emu_warp->bar);
    unsigned m = 0xFFFFFFFFu;
    for (int i = 0; i < 32; ++i) m = emu_warp->slot[i] < m ? (unsigned)emu_warp->slot[i] : m;
    pthread_barrier_wait(&emu_warp->bar);
    return m;
}
static inline int __all_sync(unsigned, int pred) { return emu_ballot(pred != 0) == 0xFFFFFFFFu; }
static inline int __any_sync(unsigned, int pred) { return emu_ballot(pred != 0) != 0u; }

// ---- launch: CTAs run one after the other (the kernels' __shared__ arrays are static), block_threads host threads that
// are created ONCE per launch and walk the grid together (a CTA-wide barrier separates consecutive CTAs): launches of
// hundreds of small CTAs no longer pay a thread creation per CUDA thread and CTA
#include <thread>
#include <tuple>
#include <vector>
template <typename... KArgs, typename... Args>
static inline void emu_launch(void (*kernel)(KArgs...), dim3 grid, unsigned block_threads, size_t smem_bytes, Args... args) {
    if (smem_bytes > emu_smem_limit(reinterpret_cast<const void *>(kernel))) {
        emu_last_error() = cudaErrorInvalidValue;
        return;
    }
    std::tuple<KArgs...> kargs(static_cast<KArgs>(args)...);
    const unsigned nwarps = (block_threads + 31) / 32;
    std::vector<EmuWarp> warps(nwarps);
    for (unsigned w = 0; w < nwarps; ++w) {
        const unsigned lanes = (w + 1) * 32 <= block_threads ? 32 : block_threads - w * 32;
        pthread_barrier_init(&warps[w].bar, nullptr, lanes);
    }
    std::vector<unsigned char> dyn(smem_bytes + 256);
    EmuCta cta;
    pthread_barrier_init(&cta.bar, nullptr, block_threads);
    cta.dyn_smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(dyn.data()) + 127) & ~(uintptr_t)127);
    std::vector<std::thread> th;
    for (unsigned t = 0; t < block_threads; ++t)
        th.emplace_back([&, t] {
            threadIdx = {t, 0, 0};
            gridDim = {grid.x, grid.y, 1};
            blockDim = {block_threads, 1, 1};
            emu_warp = &warps[t >> 5];
            emu_lane = (int)(t & 31);
            emu_cta = &cta;
            for (unsigned by = 0; by < grid.y; ++by)
                for (unsigned bx = 0; bx < grid.x; ++bx) {
                    blockIdx = {bx, by, 0};
                    std::apply(kernel, kargs);
                    pthread_barrier_wait(&cta.bar);   // the whole CTA is done before the next one reuses the shared memory
                }
        });
    for (auto &x : th) x.join();
    for (auto &w : warps) pthread_barrier_destroy(&w.bar);
    pthread_barrier_destroy(&cta.bar);
}

// ---- mbarrier + 1-D bulk copies, emulated ADVERSARIALLY --------------------------------------------------------------
// On the GPU an async bulk copy lands at some point between its issue and the completion its waiter observes.  The
// emulation takes both extremes at once: at issue time the destination is POISONED (a late reader of the old contents
// sees garbage, and ThreadSanitizer sees the write), and the real data arrives only when the first waiter polls the
// barrier (an early reader of the new contents sees poison).  Stores shared -> global are deferred likewise: the bytes
// leave shared memory only when bulk_wait_read<N>() says the group has been read, so a buffer reused too early
// corrupts the output.  mbarriers are a phase counter in the barrier's own 64-bit word.
#include <mutex>
#include <unordered_map>
#include <vector>

namespace dsk {
struct EmuPendingCopy { void *dst; const void *src; uint32_t bytes; };
struct EmuAsync {
    std::mutex mu;
    std::unordered_map<uint64_t *, EmuPendingCopy> g2s;   // keyed by the mbarrier that will signal completion
};
inline EmuAsync &emu_async() { static EmuAsync a; return a; }

static inline std::atomic<uint64_t> *emu_bar(uint64_t *bar) { return reinterpret_cast<std::atomic<uint64_t> *>(bar); }
static inline void mbar_init(uint64_t *bar, uint32_t) {
    std::lock_guard<std::mutex> lk(emu_async().mu);
    emu_async().g2s.erase(bar);
    emu_bar(bar)->store(0, std::memory_order_release);
}
static inline void fence_mbar_init() {}
static inline void fence_proxy_async() {}
static inline void mbar_arrive_expect_tx(uint64_t *, uint32_t) {}   // the phase completes when the copy is delivered
static inline void mbar_arrive(uint64_t *bar) { emu_bar(bar)->fetch_add(1, std::memory_order_release); }
static inline bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    if ((emu_bar(bar)->load(std::memory_order_acquire) & 1u) != parity) return true;
    {
        std::lock_guard<std::mutex> lk(emu_async().mu);
        auto it = emu_async().g2s.find(bar);
        if (it != emu_async().g2s.end()) {            // deliver the copy now: the latest moment the hardware could
            memcpy(it->second.dst, it->second.src, it->second.bytes);
            emu_async().g2s.erase(it);
            emu_bar(bar)->fetch_add(1, std::memory_order_release);
            return true;
        }
    }
    sched_yield();
    return false;
}
static inline void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
static inline void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    memset(dst, 0xA5, bytes);                          // the earliest moment: the old contents are gone
    std::lock_guard<std::mutex> lk(emu_async().mu);
    emu_async().g2s[bar] = EmuPendingCopy{dst, src, bytes};
}

// shared -> global bulk stores: per issuing thread, grouped by bulk_commit(), drained by bulk_wait_read<N>()
struct EmuStoreQueue { std::vector<std::vector<EmuPendingCopy>> groups; std::vector<EmuPendingCopy> open; };
inline EmuStoreQueue &emu_stores() { static thread_local EmuStoreQueue q; return q; }
static inline void bulk_s2g(void *dst, const void *src, uint32_t bytes) { emu_stores().open.push_back({dst, src, bytes}); }
static inline void bulk_commit() {
    emu_stores().groups.push_back(std::move(emu_stores().open));
    emu_stores().open.clear();
}
template <int N>
static inline void bulk_wait_read() {   // all but the newest N groups have been read out of shared memory
    auto &g = emu_stores().groups;
    while ((int)g.size() > N) {
        for (const auto &c : g.front()) memcpy(c.dst, c.src, c.bytes);
        g.erase(g.begin());
    }
}
static inline uint32_t umin3(uint32_t a, uint32_t b, uint32_t c) { return min(min(a, b), c); }
}  // namespace dsk
