// engine.h — context and scratch-arena definitions shared by the translation units of libb200trie.so.
#pragma once
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/b200trie.h"
#include "pinned_pool.h"

// ------------------------------------------------------------------------------------------------ context
// One device allocation, charged to its owner's byte counter (a context's, a resident trie's, a dynamic trie's or state's)
// for as long as it lives.  Move-only: a move hands the allocation to the destination and its bytes to the destination's
// counter.  Both grow operations do nothing while `need` bytes fit and otherwise allocate `want` bytes; the old allocation
// is freed only after `st` has drained, because work queued there may still use it.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;

    DevBuf(uint64_t *counter) : counter_(counter) {}
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap), counter_(o.counter_) {
        o.p = nullptr;
        o.cap = 0;
    }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) {
            reset();
            *o.counter_ -= o.cap;
            *counter_ += o.cap;
            p = o.p;
            cap = o.cap;
            o.p = nullptr;
            o.cap = 0;
        }
        return *this;
    }
    ~DevBuf() { reset(); }

    void reset() {
        if (p) {
            cudaFree(p);
            *counter_ -= cap;
        }
        p = nullptr;
        cap = 0;
    }
    // contents dropped: the old allocation is freed before the new one is made
    cudaError_t grow(size_t need, size_t want, cudaStream_t st) {
        if (need <= cap) return cudaSuccess;
        void *np = nullptr;
        cudaError_t e = free_after(st);
        if (e == cudaSuccess) e = cudaMalloc(&np, want);
        if (e != cudaSuccess) return e;
        p = np;
        cap = want;
        *counter_ += want;
        return cudaSuccess;
    }
    // the first `keep` bytes move to the new allocation; fill >= 0 sets every other byte to `fill`
    cudaError_t grow_keep(size_t need, size_t want, size_t keep, int fill, cudaStream_t st) {
        if (need <= cap) return cudaSuccess;
        DevBuf nb(counter_);
        cudaError_t e = nb.grow(want, want, st);
        if (e == cudaSuccess && fill >= 0) e = cudaMemsetAsync(nb.p, fill, want, st);
        if (e == cudaSuccess && p && keep) e = cudaMemcpyAsync(nb.p, p, keep, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = free_after(st);
        if (e == cudaSuccess) *this = std::move(nb);
        return e;
    }

  private:
    uint64_t *counter_;
    cudaError_t free_after(cudaStream_t st) {
        if (!p) return cudaSuccess;
        cudaError_t e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = cudaFree(p);
        if (e != cudaSuccess) return e;
        *counter_ -= cap;
        p = nullptr;
        cap = 0;
        return cudaSuccess;
    }
};
// Owned<T>: a handle released by its destroy function when it goes out of scope (seed tries, half-built handles)
template <class T>
using Owned = std::unique_ptr<T, void (*)(T *)>;

struct b200_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_streams[3] = {nullptr, nullptr, nullptr};
    // structure pass of a build (sorts, scans, flags: memory / latency bound) runs here, next to the ALU-bound leaf pass
    // on `stream`; highest priority, so that its short kernels get the SM slots the leaf pass frees
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> chunk_events;
    std::mutex mu;
    std::mutex err_mu;  // guards err: argument checks report errors before they take `mu`
    std::string err;
    uint64_t dev_bytes = 0;  // what every DevBuf below is charged to
    unsigned launches = 0;
    b200_stats stats{};
    bool stats_pending = false;
    bool stats_wavefront = false;  // branches_added of the last build comes from the wavefront's node counter
    uint64_t extra_blocks = 0;     // rate blocks beyond the first of the branch nodes built since reset_build_state
    bool extra_blocks_valid = false;  // every node of this call went through build_forest's class histogram
    // scratch (grow-only)
    DevBuf Lp{&dev_bytes}, nibs{&dev_bytes}, leaf_ref{&dev_bytes}, leaf_meta{&dev_bytes}, S{&dev_bytes}, E{&dev_bytes},
        iota{&dev_bytes}, depth_sorted{&dev_bytes}, gap_sorted{&dev_bytes}, head{&dev_bytes}, node_start{&dev_bytes},
        node_ref{&dev_bytes}, node_meta{&dev_bytes}, node_l{&dev_bytes}, node_r{&dev_bytes}, node_masks{&dev_bytes},
        cub_temp{&dev_bytes}, small{&dev_bytes}, sroots{&dev_bytes}, buckets{&dev_bytes};
    DevBuf upd_flags{&dev_bytes}, upd_nh{&dev_bytes}, upd_ids{&dev_bytes}, upd_prefix{&dev_bytes}, upd_key{&dev_bytes},
        upd_key2{&dev_bytes}, upd_ids2{&dev_bytes};
    DevBuf sort_ka{&dev_bytes}, sort_kb{&dev_bytes}, sort_ia{&dev_bytes}, sort_flag{&dev_bytes}, sort_perm{&dev_bytes},
        sort_out{&dev_bytes};
    // composite sort: sorted address digests, their permutation, head flags / dense ranks, rank by address
    DevBuf sort_aux[4]{&dev_bytes, &dev_bytes, &dev_bytes, &dev_bytes};
    DevBuf node_key{&dev_bytes}, node_key2{&dev_bytes}, node_ids{&dev_bytes}, node_order{&dev_bytes};
    // ordered tries (eng_ordered.inl)
    DevBuf ord_keys{&dev_bytes}, ord_knib{&dev_bytes}, ord_item{&dev_bytes}, ord_sched{&dev_bytes},
        ord_sched2{&dev_bytes}, ord_pos{&dev_bytes}, ord_order{&dev_bytes};
    // staging for host-pointer entry points
    DevBuf in_a{&dev_bytes}, in_b{&dev_bytes}, in_c{&dev_bytes}, in_d{&dev_bytes}, in_e{&dev_bytes}, out_a{&dev_bytes};
    DevBuf chunk_in[3]{&dev_bytes, &dev_bytes, &dev_bytes}, chunk_out[3]{&dev_bytes, &dev_bytes, &dev_bytes};
    void *pinned_small = nullptr;  // 4 KiB page-locked readback area
    // B200_PHASE_TIMING=1 (development aid): CUDA events at the phase boundaries of a build, reported by b200_sync on stderr
    bool phase_timing = false;
    std::vector<std::pair<const char *, cudaEvent_t>> phases;
    std::vector<cudaEvent_t> phase_pool;
};

inline void phase_mark(b200_ctx *c, const char *name) {
    if (!c->phase_timing) return;
    cudaEvent_t ev = nullptr;
    if (!c->phase_pool.empty()) {
        ev = c->phase_pool.back();
        c->phase_pool.pop_back();
    } else if (cudaEventCreate(&ev) != cudaSuccess) {
        return;
    }
    cudaEventRecord(ev, c->stream);
    c->phases.emplace_back(name, ev);
}
inline void phase_report(b200_ctx *c) {  // after a stream synchronize
    if (c->phases.size() > 1) {
        float total = 0;
        cudaEventElapsedTime(&total, c->phases.front().second, c->phases.back().second);
        fprintf(stderr, "[b200 phases] total %.3f ms:", total);
        for (size_t i = 1; i < c->phases.size(); i++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, c->phases[i - 1].second, c->phases[i].second);
            fprintf(stderr, " %s %.3f", c->phases[i].first, ms);
        }
        fprintf(stderr, "\n");
    }
    for (auto &p : c->phases) c->phase_pool.push_back(p.second);
    c->phases.clear();
}

inline int32_t fail(b200_ctx *c, int32_t code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) {
        std::lock_guard<std::mutex> g(c->err_mu);
        c->err = buf;
    }
    return code;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return fail(c, e__ == cudaErrorMemoryAllocation ? B200_ERR_OOM : B200_ERR_CUDA, "%s: %s (%s:%d)", \
                        #call, cudaGetErrorString(e__), __FILE__, __LINE__);                                  \
    } while (0)

// context scratch: slack so that slowly growing inputs do not re-allocate every call
inline size_t ctx_scratch_bytes(size_t bytes) { return bytes + bytes / 8 + 256; }
inline int32_t ensure(b200_ctx *c, DevBuf &b, size_t bytes) {
    CU(b.grow(bytes, ctx_scratch_bytes(bytes), c->stream));
    return B200_OK;
}
#define ENSURE(buf, bytes)                                   \
    do {                                                     \
        int32_t r__ = ensure(c, c->buf, (size_t)(bytes));    \
        if (r__ != B200_OK) return r__;                      \
    } while (0)
#define TRY(expr)                         \
    do {                                  \
        int32_t r__ = (expr);             \
        if (r__ != B200_OK) return r__;   \
    } while (0)

