// nr_internal.h -- the host-side services every host translation unit uses (context, error reporting, 2-bit packing,
// the caching allocator and what is built on them).  Not part of the C ABI.  Kernel translation units (nr_launch_*.cu)
// must not include it: their code placement follows the exact text they are compiled from (DESIGN.md section 9).
#pragma once
#include "../../include/nanorepeat_b200.h"
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

namespace nri {
int ensure_init();                               // lazy CUDA initialisation; sets this thread's device
cudaStream_t stream();                           // the library's stream
int sm_count();
int fail(int code, const char* fmt, ...)         // records the thread's last error (nr_last_error), returns code
    __attribute__((format(printf, 2, 3)));
int last_code();
bool pack(const char* s, int len, uint32_t* w);  // 16 bases per word, MSB first; false: a base other than ACGT was seen
void ambiguity(const char* s, int len, uint32_t* m);   // bit plane of the bases that are not ACGT
int alloc(void** p, size_t bytes, bool pinned);
void release(void* p, size_t bytes, bool pinned);
int check(const nr_scoring_t* sc);
void set_last_stats(const nr_stats_t& st);       // what nr_last_stats reports on this thread

constexpr int kMaxScore = 32767;   // signed 16-bit score field of the packed DP word

// A failed CUDA call: record "<call> failed: <error> (<file>:<line>)" and return NR_ERR_CUDA.  The error is cleared, so
// that it cannot be picked up again by the next launch's check.
#define CUDA_TRY(expr)                                                                                            \
    do {                                                                                                          \
        const cudaError_t e__ = (expr);                                                                           \
        if (e__ != cudaSuccess) {                                                                                 \
            cudaGetLastError();                                                                                   \
            return nri::fail(NR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
        }                                                                                                         \
    } while (0)

// Device and pinned buffers of one call, given back to the caching allocator on scope exit.  Every buffer holds at least
// 16 bytes (the allocator hands out whole size classes anyway), so an empty one needs no special case.
struct Bufs {
    struct One { void* p; size_t bytes; bool pinned; };
    std::vector<One> all;
    int get(void** p, size_t bytes, bool pinned) {
        if (bytes < 16) bytes = 16;
        *p = nullptr;
        const int rc = alloc(p, bytes, pinned);
        if (rc == NR_OK) all.push_back({*p, bytes, pinned});
        return rc;
    }
    ~Bufs() { for (const One& b : all) release(b.p, b.bytes, b.pinned); }
};

// Sequence pool.  Every sequence starts on a word boundary and is followed by one slack word (kernels prefetch one word
// ahead).  For a READ the slack word doubles as the link to its ambiguity plane: 0 = ACGT only, otherwise the plane
// starts that many words behind the read's first word (nr_kernels.cuh, read_has_ambiguous).  Templates must be ACGT.
struct Pool {
    std::vector<uint32_t> words;
    // append; returns first word index, or -1 on a non-ACGT character (ambiguous_ok: append the plane instead)
    long long add(const char* s, int len, bool ambiguous_ok = false) {
        const size_t w0 = words.size();
        const size_t nw = (size_t)(len + 15) / 16 + 1;
        words.resize(w0 + nw, 0u);
        if (!pack(s, len, words.data() + w0)) {
            if (!ambiguous_ok) { words.resize(w0); return -1; }
            link_plane(w0, s, len);
        }
        return (long long)w0;
    }
    // append the ambiguity plane of the read packed at word w0 and link it from the read's slack word
    void link_plane(size_t w0, const char* s, int len) {
        const size_t at = words.size();
        words.resize(at + (size_t)(len + 31) / 32, 0u);
        ambiguity(s, len, words.data() + at);
        words[w0 + (size_t)(len + 15) / 16] = (uint32_t)(at - w0);
    }
};

// NR_TRACE=1: host-side phase times of a call on stderr (where a call's half millisecond goes)
struct PhaseTrace {
    const bool on = getenv("NR_TRACE") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void mark(const char* what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[nr trace] %-28s %8.1f us   (ends at %10.1f us, thread %04x)\n", what,
                std::chrono::duration<double, std::micro>(t1 - t0).count(), std::fmod(std::chrono::duration<double, std::micro>(t1.time_since_epoch()).count(), 1e8),
                (unsigned)(std::hash<std::thread::id>()(std::this_thread::get_id()) & 0xffff));
        t0 = t1;
    }
};

}  // namespace nri
