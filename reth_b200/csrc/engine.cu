// engine.cu — context, HBM scratch arena, build orchestration and the extern "C" B200_API boundary of
// libb200trie.so (include/b200trie.h).  No CPU fallback exists: every entry point needs a CUDA device.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#if defined(__linux__)
#ifndef _GNU_SOURCE
#define _GNU_SOURCE
#endif
#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>
#endif

#include <algorithm>
#include <cctype>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "engine.h"
#include "kernels.h"
#include "trie_kernels.h"

using namespace b200;

#define B200_VERSION_STR "reth_b200 0.2.0 (sm_100a)"

static thread_local int g_create_status = 0;

// levels with at most this many nodes run one warp per node (shuffle-based Keccak): beyond ~3-4k nodes the 14x higher instruction count of the shuffle formulation outweighs its ~5x shorter latency
static constexpr uint32_t WARP_LEVEL_MAX = 4096;

// layout of the `small` device buffer (uint32 units)
enum : int { SM_BUCKET_OFF = 0, SM_LEVEL_LO = 80, SM_NNODES = 160, SM_ERR = 164, SM_ERR_STICKY = 165, SM_NSTORED = 168, SM_ORD_NLONG = 170, SM_UNRESOLVED = 172, SM_COUNTERS = 176 /* 4 x u64 */, SM_HIST = 256 /* 256 x u32 */, SM_WORDS = 512 };

static uint32_t *small_u32(b200_ctx *c) { return static_cast<uint32_t *>(c->small.p); }

extern "C" B200_API int32_t b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" B200_API int32_t b200_create_status(void) { return g_create_status; }

extern "C" B200_API b200_ctx *b200_create(int32_t device_ordinal) {
    int n = b200_device_count();
    if (n <= 0 || device_ordinal < 0 || device_ordinal >= n) {
        g_create_status = n <= 0 ? B200_ERR_NO_DEVICE : B200_ERR_INVALID_ARG;
        return nullptr;
    }
    b200_ctx *c = new b200_ctx();
    c->device = device_ordinal;
    auto bail = [&](cudaError_t e) -> b200_ctx * {
        g_create_status = e == cudaErrorMemoryAllocation ? B200_ERR_OOM : B200_ERR_CUDA;
        cudaGetLastError();
        b200_destroy(c);  // releases whatever was created so far
        return nullptr;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(device_ordinal)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    c->stream = c->own_stream;
    for (int i = 0; i < 3; i++)
        if ((e = cudaStreamCreateWithFlags(&c->copy_streams[i], cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi = numerically lowest = greatest priority
        if ((e = cudaStreamCreateWithPriority(&c->aux_stream, cudaStreamNonBlocking, hi)) != cudaSuccess) return bail(e);
    }
    if ((e = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&c->ev0)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&c->ev1)) != cudaSuccess) return bail(e);
    if ((e = cudaMallocHost(&c->pinned_small, 4096)) != cudaSuccess) return bail(e);
    if ((e = c->small.grow(SM_WORDS * 4, SM_WORDS * 4, c->stream)) != cudaSuccess) return bail(e);
    if ((e = cudaMemset(c->small.p, 0, SM_WORDS * 4)) != cudaSuccess) return bail(e);
    c->phase_timing = getenv("B200_PHASE_TIMING") != nullptr;
    g_create_status = B200_OK;
    return c;
}

extern "C" B200_API void b200_destroy(b200_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    if (c->pinned_small) cudaFreeHost(c->pinned_small);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    for (cudaEvent_t e : c->chunk_events) cudaEventDestroy(e);
    for (auto &p : c->phases) cudaEventDestroy(p.second);
    for (cudaEvent_t e : c->phase_pool) cudaEventDestroy(e);
    for (int i = 0; i < 3; i++)
        if (c->copy_streams[i]) cudaStreamDestroy(c->copy_streams[i]);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;  // frees the scratch buffers
}

extern "C" B200_API const char *b200_last_error(const b200_ctx *c) {
    if (!c) return "null context";
    // a copy per calling thread: another thread's failing call may rewrite the context's string at any time
    static thread_local std::string mine;
    {
        std::lock_guard<std::mutex> g(const_cast<b200_ctx *>(c)->err_mu);
        mine = c->err;
    }
    return mine.c_str();
}
extern "C" B200_API const char *b200_version(void) { return B200_VERSION_STR; }
extern "C" B200_API uint64_t b200_device_bytes(const b200_ctx *c) { return c ? c->dev_bytes : 0; }

extern "C" B200_API int32_t b200_set_stream(b200_ctx *c, void *cuda_stream) {
    if (!c) return B200_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(c->mu);
    // 0 is the CUDA legacy default stream; "no stream given" is spelled b200_set_stream(ctx, (void*)-1)
    c->stream = cuda_stream == reinterpret_cast<void *>(-1) ? c->own_stream
                : cuda_stream == nullptr                    ? cudaStreamLegacy
                                                            : static_cast<cudaStream_t>(cuda_stream);
    return B200_OK;
}

extern "C" B200_API int32_t b200_numa_bind_thread(int32_t device_ordinal) {
#if defined(__linux__)
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device_ordinal) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    for (char *p = bus; *p; p++) *p = (char)tolower((unsigned char)*p);
    char path[160];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE *f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0 || node >= 1024) return -1;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return -1;
    cpu_set_t set;
    CPU_ZERO(&set);
    int a = 0, b = 0, any = 0;
    for (;;) {  // "0-31,64-95"
        if (fscanf(f, "%d", &a) != 1) break;
        b = a;
        int ch = fgetc(f);
        if (ch == '-') {
            if (fscanf(f, "%d", &b) != 1) break;
            ch = fgetc(f);
        }
        for (int cpu = a; cpu <= b && cpu < CPU_SETSIZE; cpu++) {
            CPU_SET(cpu, &set);
            any = 1;
        }
        if (ch != ',') break;
    }
    fclose(f);
    if (!any) return -1;
    // keep only CPUs the process may use at all (cgroup / taskset), then bind; an empty intersection changes nothing
    cpu_set_t cur, both;
    if (sched_getaffinity(0, sizeof cur, &cur) == 0) {
        CPU_AND(&both, &set, &cur);
        if (CPU_COUNT(&both) == 0) return -1;
        set = both;
    }
    if (sched_setaffinity(0, sizeof set, &set) != 0) return -1;
    unsigned long mask[16] = {0};  // MPOL_PREFERRED: fall back to other nodes rather than fail an allocation
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(8 * sizeof mask));
    return node;
#else
    (void)device_ordinal;
    return -1;
#endif
}

// ------------------------------------------------------------------------------------------------ pinned result blocks
namespace {
struct PinnedPool {
    std::mutex mu;
    std::multimap<size_t, void *> idle;          // capacity -> block
    std::unordered_map<void *, size_t> capacity;  // every block this pool has handed out or holds
    size_t idle_bytes = 0;
    size_t limit = [] {
        const char *e = getenv("B200_PINNED_POOL_MB");
        return (size_t)(e ? strtoull(e, nullptr, 10) : 1024) << 20;
    }();
};
PinnedPool &pinned_pool() {
    static PinnedPool *p = new PinnedPool();  // never destroyed: blocks may be released after static destruction began
    return *p;
}
size_t pinned_size_class(size_t bytes) {  // next multiple of an eighth of the enclosing power of two, at least 4 KiB
    if (bytes <= 4096) return 4096;
    size_t pow2 = 4096;
    while (pow2 < bytes) pow2 <<= 1;
    size_t step = pow2 >> 4;  // (pow2 / 2) / 8
    return (bytes + step - 1) / step * step;
}
}  // namespace

void *pinned_block_alloc(size_t bytes) {
    const size_t want = pinned_size_class(bytes);
    PinnedPool &pp = pinned_pool();
    {
        std::lock_guard<std::mutex> g(pp.mu);
        auto it = pp.idle.lower_bound(want);
        if (it != pp.idle.end() && it->first <= 2 * want) {
            void *p = it->second;
            pp.idle_bytes -= it->first;
            pp.idle.erase(it);
            return p;
        }
    }
    void *p = nullptr;
    if (cudaMallocHost(&p, want) != cudaSuccess) {
        cudaGetLastError();
        // pinned memory is exhausted: give the idle blocks back and try once more
        std::vector<void *> drop;
        {
            std::lock_guard<std::mutex> g(pp.mu);
            for (auto &kv : pp.idle) {
                drop.push_back(kv.second);
                pp.capacity.erase(kv.second);
            }
            pp.idle.clear();
            pp.idle_bytes = 0;
        }
        for (void *q : drop) cudaFreeHost(q);
        if (cudaMallocHost(&p, want) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
    }
    std::lock_guard<std::mutex> g(pp.mu);
    pp.capacity[p] = want;
    return p;
}

void pinned_block_free(void *p) {
    if (!p) return;
    PinnedPool &pp = pinned_pool();
    {
        std::lock_guard<std::mutex> g(pp.mu);
        auto it = pp.capacity.find(p);
        if (it != pp.capacity.end() && pp.idle_bytes + it->second <= pp.limit) {
            pp.idle.emplace(it->second, p);
            pp.idle_bytes += it->second;
            return;
        }
        if (it != pp.capacity.end()) pp.capacity.erase(it);
    }
    cudaFreeHost(p);
}

extern "C" B200_API void *b200_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" B200_API void b200_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

static int32_t map_dev_error(b200_ctx *c, int code) {
    switch (code) {
        case B200_DEVERR_NONE: return B200_OK;
        case B200_DEVERR_UNSORTED: return fail(c, B200_ERR_UNSORTED, "keys are not strictly ascending inside a trie");
        case B200_DEVERR_ZERO_VALUE: return fail(c, B200_ERR_ZERO_VALUE, "storage slot with zero value (zero means deleted)");
        case B200_DEVERR_INLINE_HASH_CHILD:
            return fail(c, B200_ERR_INLINE_HASH_CHILD, "inline (<32 byte) branch child under a hash_mask bit");
        case B200_DEVERR_BAD_OFFSETS: return fail(c, B200_ERR_INVALID_ARG, "seg_offsets must start at 0, end at n and be monotone");
        case B200_DEVERR_NOT_FOUND: return fail(c, B200_ERR_NOT_FOUND, "key not found in the resident trie");
        case B200_DEVERR_CORRUPT: return fail(c, B200_ERR_CUDA, "dynamic trie: a walk exceeded 64 hops (damaged structure)");
        default: return fail(c, B200_ERR_CUDA, "unknown device error %d", code);
    }
}

// an error word read back and reported right away (mid-call read-backs of the resident / dynamic paths): the word is
// cleared, otherwise the next build would latch it as a still unreported violation of an async call
static int32_t report_dev_error_now(b200_ctx *c, int code) {
    cudaMemsetAsync(small_u32(c) + SM_ERR, 0, 4, c->stream);
    return map_dev_error(c, code);
}

// waits for the stream, folds the timing / counters of the last build into stats, returns the sticky status
static int32_t sync_and_status(b200_ctx *c) {
    CU(cudaStreamSynchronize(c->stream));
    if (c->phase_timing) phase_report(c);
    uint32_t *ps = static_cast<uint32_t *>(c->pinned_small);
    CU(cudaMemcpyAsync(ps, small_u32(c) + SM_ERR, 8, cudaMemcpyDeviceToHost, c->stream));  // current + sticky word
    CU(cudaMemcpyAsync(ps + 8, small_u32(c) + SM_COUNTERS, 32, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(ps + 4, small_u32(c) + SM_NSTORED, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (c->stats_pending) {
        if (c->stats_wavefront) c->stats.branches_added = ps[4];
        float ms = 0;
        if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) c->stats.device_ms = ms;
        else cudaGetLastError();
        const unsigned long long *cnt = reinterpret_cast<const unsigned long long *>(ps + 8);
        c->stats.hashed_nodes = cnt[CNT_HASHED];
        c->stats.extension_nodes = cnt[CNT_EXT];
        c->stats.keccak_f = c->extra_blocks_valid ? c->stats.hashed_nodes + c->extra_blocks : 0;
        c->stats_pending = false;
    }
    // the oldest unreported violation wins; reporting clears both words (a later b200_sync returns OK again)
    int code = ps[1] ? (int)ps[1] : (int)ps[0];
    if (code) CU(cudaMemsetAsync(small_u32(c) + SM_ERR, 0, 8, c->stream));
    return map_dev_error(c, code);
}

static int32_t reset_build_state(b200_ctx *c) {
    // latches a still unreported error of the previous async build into the sticky word, then clears the error word
    // and the counters for this build
    CU(launch_latch_error(reinterpret_cast<int *>(small_u32(c) + SM_ERR), reinterpret_cast<int *>(small_u32(c) + SM_ERR_STICKY),
                          reinterpret_cast<unsigned long long *>(small_u32(c) + SM_COUNTERS), c->stream));
    c->stats = b200_stats{};
    c->stats_wavefront = false;
    c->extra_blocks = 0;
    c->extra_blocks_valid = false;
    CU(cudaEventRecord(c->ev0, c->stream));
    phase_mark(c, "start");
    return B200_OK;
}
static int32_t finish_build_state(b200_ctx *c) {
    phase_mark(c, "end");
    CU(cudaEventRecord(c->ev1, c->stream));
    c->stats_pending = true;
    return B200_OK;
}

extern "C" B200_API int32_t b200_sync(b200_ctx *c) {
    if (!c) return B200_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    return sync_and_status(c);
}
extern "C" B200_API int32_t b200_dev_status(b200_ctx *c) { return b200_sync(c); }
extern "C" B200_API int32_t b200_last_stats(b200_ctx *c, b200_stats *out) {
    if (!c || !out) return B200_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    int32_t r = sync_and_status(c);
    *out = c->stats;
    return r;
}
// number of kernel launches issued through this context (bench.py reports it as gpu_launches)
extern "C" B200_API uint64_t b200_launch_count(const b200_ctx *c) { return c ? c->launches : 0; }

#include "eng_keccak.inl"
#include "eng_build.inl"
#include "eng_updates.inl"
#include "eng_roots.inl"
#include "eng_frontier.inl"
#include "eng_stream.inl"
#include "eng_resident.inl"
#include "eng_darena.inl"
#include "eng_dtrie.inl"
#include "eng_dstate.inl"
#include "eng_proofs.inl"
#include "eng_ordered.inl"
#include "eng_items.inl"
#include "eng_comm.inl"
