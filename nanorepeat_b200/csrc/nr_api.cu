// nr_api.cu -- C ABI host side of libnanorepeat_b200.so (declared in include/nanorepeat_b200.h).
//
// Host work done here, natively: 2-bit packing of reads and templates into one sequence pool, template generation
// (round 2: left + motif*T, reference nanoRepeat_bam.py:352-354; round 3: left + motif*kmax stored once per region
// plus reverse(right), or one left + motif*k + right per distinct k in the independent mode, :474-481), task
// construction over any number of regions, cost sorting, launches of the sm_100a kernels in nr_kernels.cuh, result
// gather and the round-3 selection of nanoRepeat_bam.py:423-431.
// There is no CPU compute fallback: without a CUDA device every compute call fails with NR_ERR_CUDA.
#include "nr_batch.h"

#include <algorithm>
#if defined(__x86_64__)
#include <tmmintrin.h>
#endif
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <memory>
#include <unordered_map>
#include <vector>

using namespace nrh;

namespace {

thread_local std::string g_err;
thread_local int g_code = 0;
thread_local nr_stats_t g_last_stats = {};

}  // namespace

int nrh::fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    g_code = code;
    return code;
}

namespace {

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return fail(NR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),   \
                        __FILE__, __LINE__);                                                    \
    } while (0)

using nr::kWarpsPerBlock;

// ---- context + caching allocator -----------------------------------------------------------------------------
// Batches come and go once per region (or per group of regions); cudaMalloc / cudaMallocHost / cudaFree cost far
// more than the copies they serve, so freed buffers are kept by power-of-two size class and handed out again.
enum BufKind { BUF_DEV = 0, BUF_PIN = 1, BUF_SCRATCH = 2 };
struct BufCache {
    // free_scratch: device buffers that only ever serve as the long reads' boundary-row scratch.  They are zeroed when
    // allocated and hold nothing but tagged entries of earlier launches afterwards, so a stale word can never pass for
    // an entry of the running launch (nr_kernels.cuh, load_bnd); scratch_era[ptr] = era of the last launch that used it.
    std::unordered_map<size_t, std::vector<void*>> free_dev, free_pin, free_scratch;
    std::unordered_map<void*, long long> scratch_era;
    std::unordered_map<size_t, std::vector<void*>>& of(int kind) { return kind == BUF_PIN ? free_pin : kind == BUF_SCRATCH ? free_scratch : free_dev; }
    static size_t klass(size_t bytes) {
        size_t c = 4096;
        while (c < bytes) c <<= 1;
        return c;
    }
};

struct Context {
    bool ready = false;
    int device = -1;
    int sm_count = 0;
    int clock_khz = 0;
    cudaStream_t stream = nullptr;
    BufCache cache;
};
Context g_ctx;
std::mutex g_ctx_mu;
// 3: paired flag ladder (two reads per warp, u16x2 words), 2: flag ladder, 1: shared sweeps with full records,
// 0: every rung its own rectangle
std::atomic<int> g_ladder_mode{3};
// Launches of the 32-bit kernels, process-wide.  Launch number n tags the long reads' boundary entries with epoch
// n % 1023 + 1 (10 bits of the 16-bit tag, never 0); n / 1023 is its era (see BufCache::scratch_era).
std::atomic<long long> g_launch_no{0};
constexpr long long kEpochs = 1023;
std::atomic<int> g_timing{0};        // nr_set_timing: CUDA events around every kernel of nr_batch_run

int ensure_init(int device) {
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    if (g_ctx.ready) {
        if (device >= 0 && device != g_ctx.device)
            return fail(NR_ERR_ARG, "the library is already initialised on device %d (requested %d); call nr_shutdown() first",
                        g_ctx.device, device);
        cudaSetDevice(g_ctx.device);        // the current device is per host thread: a caller's new thread starts on device 0
        return NR_OK;
    }
    if (device < 0) {
        const char* e = getenv("NR_DEVICE");
        if (!e) e = getenv("LOCAL_RANK");
        device = e ? atoi(e) : 0;
    }
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess || n == 0)
        return fail(NR_ERR_CUDA, "no CUDA device available (%s); libnanorepeat_b200 has no CPU fallback",
                    err == cudaSuccess ? "device count 0" : cudaGetErrorString(err));
    if (device >= n)       // two ranks must never end up on one GPU silently
        return fail(NR_ERR_ARG, "device %d requested but only %d CUDA device(s) are visible", device, n);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(NR_ERR_CUDA, "device %d (%s, sm_%d%d) is not a Blackwell sm_100 part", device, prop.name,
                    prop.major, prop.minor);
    CUDA_TRY(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
    g_ctx.device = device;
    g_ctx.sm_count = prop.multiProcessorCount;
    g_ctx.clock_khz = prop.clockRate;
    g_ctx.ready = true;
    return NR_OK;
}

// give every cached free buffer back to the driver (called when an allocation fails, and by nr_shutdown)
void trim_cache_locked() {
    for (auto& kv : g_ctx.cache.free_dev) for (void* p : kv.second) cudaFree(p);
    for (auto& kv : g_ctx.cache.free_scratch) for (void* p : kv.second) { cudaFree(p); g_ctx.cache.scratch_era.erase(p); }
    for (auto& kv : g_ctx.cache.free_pin) for (void* p : kv.second) cudaFreeHost(p);
    g_ctx.cache.free_dev.clear(); g_ctx.cache.free_scratch.clear(); g_ctx.cache.free_pin.clear();
}

int cached_alloc(void** p, size_t bytes, int kind) {
    const size_t k = BufCache::klass(bytes);
    {
        std::lock_guard<std::mutex> lk(g_ctx_mu);
        auto& fl = g_ctx.cache.of(kind)[k];
        if (!fl.empty()) { *p = fl.back(); fl.pop_back(); return NR_OK; }
    }
    auto raw = [&]() { return kind == BUF_PIN ? cudaMallocHost(p, k) : cudaMalloc(p, k); };
    cudaError_t e = raw();
    if (e != cudaSuccess) {        // out of memory while the cache may hold plenty: hand the cache back and try once more
        cudaGetLastError();
        { std::lock_guard<std::mutex> lk(g_ctx_mu); cudaDeviceSynchronize(); trim_cache_locked(); }
        e = raw();
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(NR_ERR_CUDA, "%s of %zu bytes failed: %s", kind == BUF_PIN ? "cudaMallocHost" : "cudaMalloc", k, cudaGetErrorString(e));
    }
    if (kind == BUF_SCRATCH) {
        CUDA_TRY(cudaMemsetAsync(*p, 0, k, g_ctx.stream));
        CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
        std::lock_guard<std::mutex> lk(g_ctx_mu);
        g_ctx.cache.scratch_era[*p] = g_launch_no.load() / kEpochs;
    }
    return NR_OK;
}

void cached_free(void* p, size_t bytes, int kind) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    g_ctx.cache.of(kind)[BufCache::klass(bytes)].push_back(p);
}

// ---- 2-bit packing -------------------------------------------------------------------------------------------
// 2-bit code of a base: (c >> 1) & 3  ->  A/a 0, C/c 1, T/t 2, G/g 3 (any bijection does: queries and targets go
// through the same packer).  Validity comes from a table.
struct BadTable {
    uint8_t t[256];
    BadTable() {
        memset(t, 1, sizeof t);
        for (const char* p = "ACGTacgt"; *p; ++p) t[(unsigned char)*p] = 0;
    }
};
const BadTable g_bad;

#if defined(__x86_64__)
// 16 bases -> one word, and their validity: lower-case and compare with "acgt"; (c >> 1) & 3 per byte; two multiply-adds
// fold four codes into a byte (b0 * 64 + b1 * 16 + b2 * 4 + b3); a byte shuffle puts the four bytes MSB first.
__attribute__((target("ssse3"))) inline uint32_t pack16_ssse3(const unsigned char* u, unsigned& bad) {
    const __m128i v = _mm_loadu_si128(reinterpret_cast<const __m128i*>(u));
    const __m128i l = _mm_or_si128(v, _mm_set1_epi8(0x20));
    const __m128i ok = _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(l, _mm_set1_epi8('a')), _mm_cmpeq_epi8(l, _mm_set1_epi8('c'))),
                                    _mm_or_si128(_mm_cmpeq_epi8(l, _mm_set1_epi8('g')), _mm_cmpeq_epi8(l, _mm_set1_epi8('t'))));
    bad |= (unsigned)_mm_movemask_epi8(ok) ^ 0xffffu;
    const __m128i c = _mm_and_si128(_mm_srli_epi16(v, 1), _mm_set1_epi8(3));
    const __m128i p = _mm_maddubs_epi16(c, _mm_set1_epi16(0x0104));
    const __m128i q = _mm_madd_epi16(p, _mm_set1_epi32(0x00010010));
    const __m128i r = _mm_shuffle_epi8(q, _mm_set_epi8(-1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, 0, 4, 8, 12));
    return (uint32_t)_mm_cvtsi128_si32(r);
}
const bool g_have_ssse3 = __builtin_cpu_supports("ssse3");
#else
const bool g_have_ssse3 = false;
#endif

// Pack one sequence: 16 bases per 32-bit word, MSB first (base i at bits 30 - 2*(i%16) of word i/16).
// w must hold (len + 15) / 16 words.  Returns false on a character other than ACGTacgt.
bool pack_seq(const char* s, int len, uint32_t* w) {
    const unsigned char* u = reinterpret_cast<const unsigned char*>(s);
    unsigned bad = 0;
    int i = 0;
    for (; i + 16 <= len; i += 16) {
#if defined(__x86_64__)
        if (g_have_ssse3) { w[i >> 4] = pack16_ssse3(u + i, bad); continue; }
#endif
        for (int j = 0; j < 16; ++j) bad |= g_bad.t[u[i + j]];
        uint32_t v = 0;
        for (int j = 0; j < 16; ++j) v |= ((u[i + j] >> 1) & 3u) << (30 - 2 * j);
        w[i >> 4] = v;
    }
    if (i < len) {
        uint32_t v = 0;
        for (int j = 0; i + j < len; ++j) {
            bad |= g_bad.t[u[i + j]];
            v |= ((u[i + j] >> 1) & 3u) << (30 - 2 * j);
        }
        w[i >> 4] = v;
    }
    return bad == 0;
}

// Bit plane of the bases of s that are not ACGT (bit i & 31 of word i >> 5); m holds (len + 31) / 32 zeroed words.
void ambiguity_plane(const char* s, int len, uint32_t* m) {
    for (int i = 0; i < len; ++i)
        if (g_bad.t[(unsigned char)s[i]]) m[i >> 5] |= 1u << (i & 31);
}

// fn(i) for i in [0, n) on a few host threads (packing thousands of reads is the host's largest cost per call)
template <class F>
void parallel_for(int n, int grain, F fn) {
    // one process per GPU shares the host cores with its siblings (torchrun exports LOCAL_WORLD_SIZE)
    static const int share = [] { const char* e = getenv("LOCAL_WORLD_SIZE"); return e && atoi(e) > 0 ? atoi(e) : 1; }();
    int nt = (int)std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency() / (unsigned)share), 8u);
    nt = std::min(nt, std::max(1, n / std::max(1, grain)));
    if (nt <= 1) { for (int i = 0; i < n; ++i) fn(i); return; }
    std::vector<std::thread> th;
    th.reserve(nt - 1);
    auto body = [&](int t) { for (int i = (int)((long long)n * t / nt), e = (int)((long long)n * (t + 1) / nt); i < e; ++i) fn(i); };
    for (int t = 1; t < nt; ++t) th.emplace_back(body, t);
    body(0);
    for (auto& x : th) x.join();
}


// shared memory per warp, in int4: query profile (+ backward junction vectors for the ladder kernel)
int exact_smem_int4(int R) { return 4 * ((R + 3) / 4) * 32; }
int ladder_smem_int4(int R) { return exact_smem_int4(R) + R * 32; }
// paired ladder: the junction vectors are three 4-byte planes (nr_pair_kernels.cuh); the fused launch's 32-bit entries
// (at most kMaxRLadder rows per lane) need the int4 layout
int pair_ladder_smem_int4(int pair_R, int rest_R) { return std::max(exact_smem_int4(pair_R) + 3 * pair_R * 8, rest_R ? ladder_smem_int4(rest_R) : 0); }

int check_scoring(const nr_scoring_t* sc) {
    if (!sc) return fail(NR_ERR_ARG, "scoring is NULL");
    if (sc->match <= 0 || sc->mismatch < 0 || sc->gap_open1 < 0 || sc->gap_ext1 <= 0 || sc->gap_open2 < 0 ||
        sc->gap_ext2 <= 0)
        return fail(NR_ERR_ARG, "scoring values out of range");
    if (sc->ambiguous < 0 || sc->ambiguous > 4096) return fail(NR_ERR_ARG, "scoring values out of range");
    if (sc->gap_open1 + sc->gap_ext1 > 4096 || sc->gap_open2 + sc->gap_ext2 > 4096 || sc->mismatch > 4096 ||
        sc->match > 4096)
        return fail(NR_ERR_ARG, "scoring values too large for the packed kernels");
    return NR_OK;
}

nr::ScoreW score_words(const nr_scoring_t& sc) {
    nr::ScoreW k;
    k.sub_match = (sc.match << 16) - 1;
    k.sub_mismatch = -(sc.mismatch << 16) - 1;
    k.sub_amb = -(sc.ambiguous << 16) - 1;
    k.h_open1 = -((sc.gap_open1 + sc.gap_ext1) << 16) - 1;
    k.h_ext1 = -(sc.gap_ext1 << 16) - 1;
    k.h_open2 = -((sc.gap_open2 + sc.gap_ext2) << 16) - 1;
    k.h_ext2 = -(sc.gap_ext2 << 16) - 1;
    k.v_open1 = -((sc.gap_open1 + sc.gap_ext1) << 16);
    k.v_ext1 = -(sc.gap_ext1 << 16);
    k.v_open2 = -((sc.gap_open2 + sc.gap_ext2) << 16);
    k.v_ext2 = -(sc.gap_ext2 << 16);
    k.refund1 = sc.gap_open1 << 16;
    k.refund2 = sc.gap_open2 << 16;
    k.one = 1;
    k.mone = -1;
    k.four = 4u;
    k.min_score = std::max(1, sc.min_dp_score);
    return k;
}

// Allocates the buffers plan_batch sized, stages the blob's sections in pinned memory and uploads them on the library's
// stream (asynchronously: nr_batch_run orders itself behind ev_uploaded).
int upload_batch(nr_batch* b) {
    PhaseTrace trace;
    int rc;
    if ((rc = cached_alloc(&b->d_blob, b->blob_bytes, BUF_DEV))) return rc;
    if ((rc = cached_alloc(&b->h_blob, b->blob_bytes, BUF_PIN))) return rc;
    if ((rc = cached_alloc((void**)&b->d_out, b->out_bytes, BUF_DEV))) return rc;
    if ((rc = cached_alloc((void**)&b->h_out, b->out_bytes, BUF_PIN))) return rc;
    if (b->scratch_bytes && (rc = cached_alloc((void**)&b->d_scratch, b->scratch_bytes, BUF_SCRATCH))) return rc;
    if (b->flags_bytes && (rc = cached_alloc((void**)&b->d_flags, b->flags_bytes, BUF_DEV))) return rc;
    if (b->state_bytes && (rc = cached_alloc((void**)&b->d_state, b->state_bytes, BUF_DEV))) return rc;
    if (b->round2_exit &&
        (rc = cached_alloc((void**)&b->d_kept, sizeof(uint32_t) * 128 * kWarpsPerBlock * (size_t)g_ctx.sm_count, BUF_DEV))) return rc;
    if (b->flag) {
        if ((rc = cached_alloc((void**)&b->d_sel, b->sel_bytes, BUF_DEV))) return rc;
        if ((rc = cached_alloc((void**)&b->h_sel, b->sel_bytes, BUF_PIN))) return rc;
    }
    if (!b->pairs3.empty()) {
        if ((rc = cached_alloc((void**)&b->d_prung, b->prung_bytes, BUF_DEV))) return rc;
        if ((rc = cached_alloc((void**)&b->d_redo, b->redo_bytes, BUF_DEV))) return rc;
        if ((rc = cached_alloc((void**)&b->h_redo_count, 64, BUF_PIN))) return rc;
        b->h_redo_count[0] = b->h_redo_count[1] = 0;
    }
    trace.mark("buffers (cached alloc)");
    char* h = static_cast<char*>(b->h_blob);
    char* d = static_cast<char*>(b->d_blob);
    for (const Section& s : b->blob) {
        if (s.bytes) memcpy(h + s.off, s.src, s.bytes);
        memset(h + s.off + s.bytes, 0, s.zeros);
    }
    memset(h + b->blob_bytes - 256, 0, 256);
    b->d_tasks = reinterpret_cast<nr::Task*>(d + b->blob[SEC_TASKS].off);
    b->d_ltasks = reinterpret_cast<nr::LadderTask*>(d + b->blob[SEC_TASKS].off);
    b->d_lregs = reinterpret_cast<nr::LadderRegion*>(d + b->blob[SEC_LREGS].off);
    b->d_order = reinterpret_cast<int32_t*>(d + b->blob[SEC_ORDER].off);
    b->d_pairs = d + b->blob[SEC_PAIRS].off;
    b->d_coop = reinterpret_cast<nr::CoopInfo*>(d + b->blob[SEC_COOP].off);
    b->d_coop_idx = reinterpret_cast<int32_t*>(d + b->blob[SEC_COOP_IDX].off);
    b->d_pool = reinterpret_cast<uint32_t*>(d + b->blob[SEC_POOL].off);
    b->d_counters = reinterpret_cast<int*>(d + b->blob_bytes - 256);
    trace.mark("blob staging (memcpy)");
    cudaStream_t st = g_ctx.stream;
    CUDA_TRY(cudaMemcpyAsync(d, h, b->blob_bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(b->d_out, 0, b->out_bytes, st));
    if (b->d_sel) CUDA_TRY(cudaMemsetAsync(b->d_sel, 0, b->sel_bytes, st));
    CUDA_TRY(cudaEventRecord(b->ev_uploaded, st));      // nr_batch_run on another stream waits for it; no host sync here
    trace.mark("upload + memsets (async)");
    b->committed = true;
    return NR_OK;
}

int commit_batch(nr_batch* b) {
    const int rc = plan_batch(b, g_ctx.sm_count);
    return rc ? rc : upload_batch(b);
}

constexpr int kSpinSlot = 16;        // d_counters[kSpinSlot]: the batch's give-up flag (nr_kernels.cuh, wait_cols)

// Arguments of one launch of the 32-bit kernels.  Draws the launch's epoch; a scratch buffer that was last used in an
// earlier era is zeroed first (on the launch's stream), so no tag left in it can equal one of this launch.
int rest_args(nr_batch* b, const int32_t* order, int count, cudaStream_t st, nr::RestArgs* out) {
    nr::RestArgs ra;
    ra.order = order; ra.n_order = count;
    ra.scratch = b->d_scratch; ra.coop = b->d_coop; ra.coop_idx = b->d_coop_idx; ra.flags = b->d_flags;
    ra.spin = b->d_counters + kSpinSlot;
    ra.redo_long = b->d_redo ? b->d_redo + b->ltasks.size() : nullptr;
    ra.redo_long_count = b->d_counters + 4;
    const long long no = g_launch_no.fetch_add(1);
    ra.epoch = (int)(no % kEpochs) + 1;
    if (b->d_scratch) {
        bool stale;
        {
            std::lock_guard<std::mutex> lk(g_ctx_mu);
            long long& era = g_ctx.cache.scratch_era[b->d_scratch];
            stale = era != no / kEpochs;
            era = no / kEpochs;
        }
        if (stale) CUDA_TRY(cudaMemsetAsync(b->d_scratch, 0, b->scratch_bytes, st));
    }
    *out = ra;
    return NR_OK;
}

// launch of the 32-bit kernels over order[0, count) (count_dev != NULL: the count is read on the device)
int launch_rest(nr_batch* b, cudaStream_t st, const nr::ScoreW& k, const int32_t* order, int count, int blocks,
                int R, const int* count_dev, int* counter) {
    const Launch& L = b->launch;
    nr::RestArgs ra;
    int rc;
    if ((rc = rest_args(b, order, count, st, &ra))) return rc;
    if (L.ladder) {
        if (!L.fixed) return fail(NR_ERR_ARG, "the ladder kernels are built for map-ont scoring only");
        const int stride = ladder_smem_int4(R);
        // single stripes of more than 384 rows (the paired kernel's redo reads) need 16 KB per warp: fewer warps per block
        int wpb = kWarpsPerBlock;
        while (wpb > 4 && (size_t)wpb * stride * sizeof(int4) > nrl::kMaxDynShared) wpb -= 4;
        const size_t smem = (size_t)wpb * stride * sizeof(int4);
        if (smem > nrl::kMaxDynShared) return fail(NR_ERR_ARG, "launch needs %zu bytes of shared memory", smem);
        CUDA_TRY(nrl::launch_ladder(b->flag, blocks, wpb * 32, smem, st, b->d_ltasks, ra, count_dev,
                                    b->qsrc ? b->qsrc->d_pool : b->d_pool, b->d_pool, b->d_lregs, k, counter, stride, b->d_out, b->d_sel));
    } else {
        const int stride = exact_smem_int4(R);
        const size_t smem = (size_t)kWarpsPerBlock * stride * sizeof(int4);
        if (smem > nrl::kMaxDynShared) return fail(NR_ERR_ARG, "launch needs %zu bytes of shared memory", smem);
        CUDA_TRY(nrl::launch_exact(L.fixed, blocks, kWarpsPerBlock * 32, smem, st, b->d_tasks, ra, b->d_pool, k, counter, stride, b->d_out));
    }
    return NR_OK;
}

// A stream of the calling thread's own for launches without cooperating stripes.  Two nr_estimate_regions calls on two
// threads then overlap on the GPU block by block: as the persistent blocks of one call's kernel run out of work, the
// other call's blocks take their SMs, instead of the whole second kernel waiting behind the first one's tail on the
// library's one stream.  Launches WITH cooperating stripes (long reads) stay on the library's stream: their blocks wait
// for one another, so two of them must never share the GPU half-resident each.
thread_local cudaStream_t t_aux_stream = nullptr;
cudaStream_t aux_stream_for(const nr_batch* b) {
    static const bool off = getenv("NR_ONE_STREAM") != nullptr;
    if (off || !b->coop.empty()) return nullptr;
    if (!t_aux_stream && cudaStreamCreateWithFlags(&t_aux_stream, cudaStreamNonBlocking) != cudaSuccess) {
        cudaGetLastError();
        t_aux_stream = nullptr;
    }
    return t_aux_stream;
}

int run_batch(nr_batch* b, cudaStream_t st) {
    if (!b->committed) return fail(NR_ERR_ARG, "batch was not committed");
    b->run_stream = st;
    const Launch& L = b->launch;
    const nr::ScoreW k = score_words(b->sc);
    if (st != g_ctx.stream) {                 // the upload (and the reused round-2 pool's) ran on the library's stream
        CUDA_TRY(cudaStreamWaitEvent(st, b->ev_uploaded, 0));
        if (b->qsrc) CUDA_TRY(cudaStreamWaitEvent(st, b->qsrc->ev_uploaded, 0));
    }
    bool resumes = false;
    for (const nr::pr::Pair3& p : b->pairs3) resumes = resumes || p.state_off >= 0;
    if (resumes) {
        // forward sweeps take over the DP state the round-2 batch's kernel kept: it must have run, and be done first
        if (!b->qsrc->ran) return fail(NR_ERR_ARG, "nr_batch_run: the round-2 batch this round-3 batch resumes from has not been run");
        if (b->qsrc->run_stream != st) CUDA_TRY(cudaStreamWaitEvent(st, b->qsrc->ev_done, 0));
    }
    // counters: [0] main launch, [2] length of the redo list, [3] redo launch, [kSpinSlot] the long reads' give-up flag
    CUDA_TRY(cudaMemsetAsync(b->d_counters, 0, 32 * sizeof(int), st));
    if (b->flags_bytes) CUDA_TRY(cudaMemsetAsync(b->d_flags, 0, b->flags_bytes, st));
    int launches = 0;
    int rc;
    const bool timing = g_timing.load() != 0;
    if (timing)
        for (cudaEvent_t& e : b->ev_t)
            if (!e) CUDA_TRY(cudaEventCreate(&e));
    b->timed[0] = b->timed[1] = b->timed[2] = false;
    auto mark = [&](int i, cudaStream_t s) { return timing ? cudaEventRecord(b->ev_t[i], s) : cudaSuccess; };
    if (L.n_pairs || b->n_long_pairs) {
        // one persistent launch: the batch's 32-bit entries (long reads cut into stripes, ...) first, then its pairs
        const bool ladder_batch = L.ladder;
        nr::RestArgs ra;
        if ((rc = rest_args(b, b->d_order, L.count, st, &ra))) return rc;
        int wpb = kWarpsPerBlock;
        if (const char* e = getenv("NR_WPB")) wpb = std::max(4, std::min(kWarpsPerBlock, atoi(e)));   // tuning
        const int blocks = std::max(1, std::min(g_ctx.sm_count, L.count + L.n_pairs));
        nr::pr::Deal deal = nr::pr::make_deal(L.count, L.n_pairs, wpb, blocks);
        if (getenv("NR_PLAIN_DEAL")) deal.nb_long = -1;      // tuning / debugging
        CUDA_TRY(mark(2, st));
        if (!ladder_batch) {
            // the dominance exit keeps a cut (H, E1, E2 of every row) beside each pair's profile
            const int stride = std::max(exact_smem_int4(std::max(L.pair_R, L.R)),
                                        b->round2_exit ? exact_smem_int4(L.pair_R) + 3 * L.pair_R * 8 : 0);
            const size_t smem = (size_t)wpb * stride * sizeof(int4);
            if (smem > nrl::kMaxDynShared) return fail(NR_ERR_ARG, "launch needs %zu bytes of shared memory", smem);
            CUDA_TRY(nrl::launch_pair_round2(blocks, wpb * 32, smem, st, static_cast<const nr::pr::Pair2*>(b->d_pairs), deal, b->d_tasks,
                                             ra, b->d_pool, k, b->d_counters, stride, b->d_out, b->d_state, b->d_kept));
        } else {
            const int stride = pair_ladder_smem_int4(L.pair_R, L.R);
            const size_t smem = (size_t)wpb * stride * sizeof(int4);
            if (smem > nrl::kMaxDynShared) return fail(NR_ERR_ARG, "launch needs %zu bytes of shared memory", smem);
            CUDA_TRY(nrl::launch_pair_ladder(blocks, wpb * 32, smem, st, static_cast<const nr::pr::Pair3*>(b->d_pairs), deal, b->d_ltasks,
                                             ra, b->qsrc ? b->qsrc->d_pool : b->d_pool, b->d_pool, b->d_lregs, k, b->d_counters, stride,
                                             b->d_prung, b->d_out, b->d_sel, b->d_counters + 2, b->d_redo,
                                             b->qsrc ? b->qsrc->d_state : nullptr));
        }
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(mark(3, st));
        b->timed[1] = timing;
        ++launches;
        if (!b->pairs3.empty()) {
            // reads whose selection hinges on a tie the 16-bit words cannot order: 32-bit flag ladder, count on the device
            CUDA_TRY(mark(4, st));
            if ((rc = launch_rest(b, st, k, b->d_redo, 0, std::max(1, std::min(g_ctx.sm_count, 2 * L.n_pairs)), L.redo_R,
                                  b->d_counters + 2, b->d_counters + 3))) return rc;
            CUDA_TRY(mark(5, st));
            b->timed[2] = timing;
            CUDA_TRY(cudaMemcpyAsync(b->h_redo_count, b->d_counters + 2, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(b->h_redo_count + 1, b->d_counters + 4, sizeof(int), cudaMemcpyDeviceToHost, st));
            ++launches;
        }
    } else if (L.count) {
        CUDA_TRY(mark(0, st));
        if ((rc = launch_rest(b, st, k, b->d_order, L.count, L.blocks, L.R, nullptr, b->d_counters))) return rc;
        CUDA_TRY(mark(1, st));
        b->timed[0] = timing;
        ++launches;
    }
    // results start their way back as soon as the kernel is done (a fetch issued later would queue behind whatever
    // was launched on the stream in between): 16 B per task / per read; flag-ladder rung records only on request
    if (b->flag) {
        if (b->n_reads) CUDA_TRY(cudaMemcpyAsync(b->h_sel, b->d_sel, sizeof(int4) * b->n_reads, cudaMemcpyDeviceToHost, st));
    } else if (b->n_out) {
        CUDA_TRY(cudaMemcpyAsync(b->h_out, b->d_out, sizeof(int4) * b->n_out, cudaMemcpyDeviceToHost, st));
    }
    if (b->flags_bytes) {
        if (!b->h_spin) { int rc2 = cached_alloc((void**)&b->h_spin, 64, BUF_PIN); if (rc2) return rc2; }
        CUDA_TRY(cudaMemcpyAsync(b->h_spin, b->d_counters + kSpinSlot, sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaEventRecord(b->ev_done, st));
    b->stats.kernel_launches = launches;
    b->long_redone = false;
    b->ran = true;
    return NR_OK;
}

int redo_long_reads(nr_batch* b);

int fetch_raw(nr_batch* b) {
    if (!b->ran) return fail(NR_ERR_ARG, "batch was not run");
    CUDA_TRY(cudaEventSynchronize(b->ev_done));         // kernel + the copy nr_batch_run queued behind it
    if (b->h_spin && *b->h_spin)
        return fail(NR_ERR_CUDA, "a stripe of a long read gave up waiting for the stripe above it; the results of this batch are not valid");
    if (b->n_long_pairs && b->h_redo_count && b->h_redo_count[1] > 0 && !b->long_redone) return redo_long_reads(b);
    return NR_OK;
}

// A template / generic sequence.  ambiguous_ok: a query of the generic engine (bases other than ACGT are scored
// -sc_ambi through its ambiguity plane); templates must be ACGT: NR_ERR_BAD_BASE, which the region-level callers turn
// into "this region is not scored" instead of failing the batch.
int add_seq(nr_batch* b, const char* s, int len, const char* what, int idx, uint32_t* word, bool ambiguous_ok = false) {
    if (!s && len > 0) return fail(NR_ERR_ARG, "%s %d is NULL", what, idx);
    if (len < 0) return fail(NR_ERR_ARG, "%s %d has negative length", what, idx);
    long long w = b->pool.add(s, len, ambiguous_ok);
    if (w < 0) return fail(NR_ERR_BAD_BASE, "%s %d contains a character other than ACGT", what, idx);
    if (w > 0xfffffff0LL || b->pool.words.size() > 0xfffffff0ULL) return fail(NR_ERR_TOO_LARGE, "sequence pool exceeds 2^32 words");
    *word = (uint32_t)w;
    return NR_OK;
}

// reads either as an array of pointers (cores != NULL) or as one concatenated buffer with n_reads + 1 offsets
struct ReadSrc {
    const char* const* cores;
    const int32_t* core_len;
    const char* concat;
    const int64_t* off;
    int gap;        // bytes between two reads of `concat` that belong to neither (1: newline-separated lines)
    const char* ptr(int r) const { return cores ? cores[r] : concat + off[r]; }
    long long len(int r) const { return cores ? (long long)core_len[r] : (long long)(off[r + 1] - off[r] - gap); }
};

inline bool is_blank(char c) { return c == ' ' || c == '\n' || c == '\r' || c == '\t'; }

// Pack n_reads reads into the pool (in parallel); q_word[r] = first word of read r, q_len[r] its length.
// * White space around a read is not part of it: the reference writes every core to a FASTQ / FASTA file and reads it
//   back (nanoRepeat_bam.py:311-321, :487-493), which drops it.
// * A base other than ACGT is kept as an ambiguous base (minimap2's code 4, scored -sc_ambi; the reference accepts such
//   reads, only tk.rev_comp raises on them): the read gets an ambiguity plane behind the packed reads.
int add_reads(nr_batch* b, const ReadSrc& src, int n_reads, std::vector<uint32_t>& q_word, std::vector<int32_t>& q_len) {
    q_word.resize(n_reads);
    q_len.resize(n_reads);
    std::vector<const char*> ptr(n_reads);
    size_t w = b->pool.words.size();
    const size_t w0 = w;
    for (int r = 0; r < n_reads; ++r) {
        long long len = src.len(r);
        if (len < 0 || len > 0x7fffffffLL) return fail(NR_ERR_ARG, "core %d has a bad length", r);
        const char* p = src.ptr(r);
        if (len > 0 && !p) return fail(NR_ERR_ARG, "core %d is NULL", r);
        while (len > 0 && is_blank(p[len - 1])) --len;
        while (len > 0 && is_blank(*p)) { ++p; --len; }
        if (w > 0xfffffff0ULL) return fail(NR_ERR_TOO_LARGE, "sequence pool exceeds 2^32 words");
        ptr[r] = p;
        q_len[r] = (int32_t)len;
        q_word[r] = (uint32_t)w;
        w += (size_t)(len + 15) / 16 + 1;
    }
    b->pool.words.resize(w, 0u);
    uint32_t* words = b->pool.words.data();
    std::vector<uint8_t> amb(n_reads, 0);
    // ~0.1 us per read on one core
    static const int kPackGrain = [] { const char* e = getenv("NR_PACK_GRAIN"); return e && atoi(e) > 0 ? atoi(e) : 8192; }();
    parallel_for(n_reads, kPackGrain, [&](int r) { amb[r] = !pack_seq(ptr[r], q_len[r], words + q_word[r]); });
    for (int r = 0; r < n_reads; ++r)
        if (amb[r]) {
            b->pool.link_plane(q_word[r], ptr[r], q_len[r]);
            ++b->n_ambiguous_reads;
        }
    if (b->pool.words.size() > 0xfffffff0ULL) { b->pool.words.resize(w0); return fail(NR_ERR_TOO_LARGE, "sequence pool exceeds 2^32 words"); }
    return NR_OK;
}

int add_round2(nr_batch* b, const char* left, int32_t n_left, const char* motif, int32_t motif_len, int32_t T,
               int32_t n_reads, const ReadSrc& src) {
    if (!b || b->kind != KIND_ROUND2 || b->committed) return fail(NR_ERR_ARG, "not an open round-2 batch");
    if (n_left < 0 || motif_len <= 0 || T < 0 || n_reads < 0 || !motif || (n_left > 0 && !left))
        return fail(NR_ERR_ARG, "nr_batch_add_round2: bad arguments");
    const size_t pool0 = b->pool.words.size();
    // template = left + motif * T   (nanoRepeat_bam.py:352-354)
    std::string tpl(left ? left : "", (size_t)n_left);
    tpl.reserve((size_t)n_left + (size_t)motif_len * T);
    for (int k = 0; k < T; ++k) tpl.append(motif, (size_t)motif_len);
    uint32_t tw = 0;
    int rc;
    bool bad_template = false;
    if ((rc = add_seq(b, tpl.data(), (int)tpl.size(), "round-2 template", 0, &tw))) {
        if (rc != NR_ERR_BAD_BASE) return rc;
        bad_template = true;       // an anchor with N: the region is not scored (no read gets a size), the batch lives on
    }
    RegionInfo g;
    g.n_left = n_left; g.motif_len = motif_len; g.first_read = b->n_reads; g.n_reads = n_reads;
    g.left.assign(left ? left : "", (size_t)n_left);
    g.motif.assign(motif, (size_t)motif_len);
    b->regions.push_back(g);
    const size_t base = b->tasks.size();
    b->tasks.resize(base + n_reads);
    std::vector<uint32_t> qw;
    std::vector<int32_t> ql;
    if ((rc = add_reads(b, src, n_reads, qw, ql))) {     // leave the batch as it was: the caller may retry this region
        b->tasks.resize(base);
        b->regions.pop_back();
        b->pool.words.resize(pool0);
        return rc;
    }
    for (int r = 0; r < n_reads; ++r) {
        nr::Task& t = b->tasks[base + r];
        t.q_word = qw[r];
        t.q_len = ql[r];
        t.t_word = tw;
        t.t_len = bad_template ? -1 : (int)tpl.size();      // -1: not scored (plan_batch counts it as skipped)
    }
    b->n_reads += n_reads;
    return NR_OK;
}

// reuse != NULL: the reads are tasks of the round-2 batch b->qsrc (already packed, already in HBM)
int add_round3_impl(nr_batch* b, const char* left, int32_t n_left, const char* right, int32_t n_right, const char* motif,
                    int32_t motif_len, int32_t n_reads, const ReadSrc& src, const int32_t* kmin, const int32_t* kmax,
                    const nr::Task* reuse) {
    for (int r = 0; r < n_reads; ++r)
        if (kmin[r] < 0) return fail(NR_ERR_ARG, "kmin[%d] < 0", r);
    if (b->flag && 2 * (long long)n_right > 65534)
        return fail(NR_ERR_TOO_LARGE, "right anchor of %d bases exceeds the flag ladder's range (32767); use nr_set_ladder_mode(1)", n_right);
    if (reuse && !b->ladder)
        return fail(NR_ERR_ARG, "reads of a round-2 batch can only be reused by the ladder kernels (nr_set_ladder_mode 1 or 2)");
    RegionInfo g;
    g.n_left = n_left; g.n_right = n_right; g.motif_len = motif_len; g.first_read = b->n_reads; g.n_reads = n_reads;
    const int region = (int)b->regions.size();
    b->regions.push_back(g);
    if (b->rung_off.empty()) b->rung_off.push_back(0);
    int klo = INT32_MAX, khi = -1;
    for (int r = 0; r < n_reads; ++r) {
        const long long n = kmax[r] >= kmin[r] ? (long long)kmax[r] - kmin[r] + 1 : 0;
        b->rung_off.push_back(b->rung_off.back() + n);
        b->kmin.push_back(kmin[r]);
        b->kmax.push_back(kmax[r]);
        b->read_region.push_back(region);
        if (n) { klo = std::min(klo, kmin[r]); khi = std::max(khi, kmax[r]); }
    }
    if (b->rung_off.back() > 0x7fffffffLL) return fail(NR_ERR_TOO_LARGE, "more than 2^31 rungs in one batch");
    const int first = b->n_reads;
    b->n_reads += n_reads;
    b->n_out = (size_t)b->rung_off.back();
    const int64_t* roff = b->rung_off.data() + first;
    int rc;
    // a template with a base other than ACGT (an anchor with N): the region is not scored -- its reads come back with
    // top_score 0 ("minimap2 printed nothing", nanoRepeat_bam.py:421) and count as skipped; the batch lives on
    bool bad_template = false;
    std::vector<uint32_t> qw;
    std::vector<int32_t> ql;
    if (b->ladder) {
        // shared sweeps (nr_kernels.cuh, ladder_kernel): the pool holds left + motif^khi once and reverse(right) once
        nr::LadderRegion lr = {};
        lr.n_left = n_left; lr.n_right = n_right; lr.m = motif_len;
        std::string fwd(left ? left : "", (size_t)n_left);
        for (int u = 0; u < std::max(khi, 0); ++u) fwd.append(motif, (size_t)motif_len);
        std::string rev(right ? right : "", (size_t)n_right);
        std::reverse(rev.begin(), rev.end());
        if ((rc = add_seq(b, fwd.data(), (int)fwd.size(), "ladder prefix", 0, &lr.fwd_word)) ||
            (rc = add_seq(b, rev.data(), (int)rev.size(), "right anchor", 0, &lr.rev_word))) {
            if (rc != NR_ERR_BAD_BASE) return rc;
            bad_template = true;
        }
        const int lreg = (int)b->lregs.size();
        b->lregs.push_back(lr);
        if (!reuse && (rc = add_reads(b, src, n_reads, qw, ql))) return rc;
        for (int r = 0; r < n_reads; ++r) {
            if (roff[r + 1] == roff[r]) continue;
            if (bad_template) { ++b->n_skipped; continue; }
            nr::LadderTask t = {};
            if (reuse) { t.q_word = reuse[r].q_word; t.q_len = reuse[r].q_len; }
            else { t.q_word = qw[r]; t.q_len = ql[r]; }
            if (t.q_len == 0) continue;     // every rung scores 0: the outputs are zero-filled
            t.kmin = kmin[r];
            t.kmax = kmax[r];
            t.out_off = (int32_t)roff[r];
            t.region = lreg;
            t.read = first + r;
            b->ltasks.push_back(t);
            b->lt_src.push_back(reuse ? (int32_t)(reuse - b->qsrc->tasks.data()) + r : -1);
        }
        return NR_OK;
    }
    // independent rectangles: left + motif*k + right, one template per distinct k that any read of the region uses
    // (nanoRepeat_bam.py:478-479)
    std::vector<uint32_t> tpl_word;
    if (khi >= klo) {
        std::vector<uint8_t> used(khi - klo + 1, 0);
        for (int r = 0; r < n_reads; ++r)
            for (int k = kmin[r]; k <= kmax[r]; ++k) used[k - klo] = 1;
        tpl_word.assign(khi - klo + 1, 0);
        std::string tpl;
        for (int k = klo; k <= khi && !bad_template; ++k) {
            if (!used[k - klo]) continue;
            tpl.assign(left ? left : "", (size_t)n_left);
            for (int u = 0; u < k; ++u) tpl.append(motif, (size_t)motif_len);
            tpl.append(right ? right : "", (size_t)n_right);
            if ((rc = add_seq(b, tpl.data(), (int)tpl.size(), "ladder template", k, &tpl_word[k - klo]))) {
                if (rc != NR_ERR_BAD_BASE) return rc;
                bad_template = true;
            }
        }
    }
    if ((rc = add_reads(b, src, n_reads, qw, ql))) return rc;
    b->tasks.resize(b->n_out);
    for (int r = 0; r < n_reads; ++r) {
        for (int k = kmin[r]; k <= kmax[r]; ++k) {
            nr::Task& t = b->tasks[(size_t)(roff[r] + (k - kmin[r]))];
            t.q_word = qw[r];
            t.q_len = ql[r];
            t.t_word = bad_template ? 0u : tpl_word[k - klo];
            t.t_len = bad_template ? -1 : n_left + motif_len * k + n_right;      // -1: not scored (plan_batch)
        }
    }
    return NR_OK;
}

// Validates first; a failure further down (pool overflow, too many rungs) restores the batch to what it was, so the
// caller may go on adding other regions (like nr_batch_add_round2).
int add_round3(nr_batch* b, const char* left, int32_t n_left, const char* right, int32_t n_right, const char* motif,
               int32_t motif_len, int32_t n_reads, const ReadSrc& src, const int32_t* kmin, const int32_t* kmax,
               const nr::Task* reuse = nullptr) {
    if (!b || b->kind != KIND_ROUND3 || b->committed) return fail(NR_ERR_ARG, "not an open round-3 batch");
    if (n_left < 0 || n_right < 0 || motif_len <= 0 || n_reads < 0 || !motif || (n_left > 0 && !left) ||
        (n_right > 0 && !right) || (n_reads > 0 && (!kmin || !kmax)))
        return fail(NR_ERR_ARG, "nr_batch_add_round3: bad arguments");
    const size_t n_regions = b->regions.size(), n_roff = b->rung_off.size(), n_k = b->kmin.size(), n_rr = b->read_region.size(),
                 n_lregs = b->lregs.size(), n_lt = b->ltasks.size(), n_src = b->lt_src.size(), n_tasks = b->tasks.size(),
                 n_words = b->pool.words.size(), n_out = b->n_out;
    const int n_reads0 = b->n_reads, n_skipped0 = b->n_skipped, n_amb0 = b->n_ambiguous_reads;
    const int rc = add_round3_impl(b, left, n_left, right, n_right, motif, motif_len, n_reads, src, kmin, kmax, reuse);
    if (rc) {
        b->regions.resize(n_regions); b->rung_off.resize(n_roff); b->kmin.resize(n_k); b->kmax.resize(n_k);
        b->read_region.resize(n_rr); b->lregs.resize(n_lregs); b->ltasks.resize(n_lt); b->lt_src.resize(n_src);
        b->tasks.resize(n_tasks); b->pool.words.resize(n_words);
        b->n_out = n_out; b->n_reads = n_reads0; b->n_skipped = n_skipped0; b->n_ambiguous_reads = n_amb0;
    }
    return rc;
}

void free_events(nr_batch* b) {
    for (cudaEvent_t* e : {&b->ev_uploaded, &b->ev_done, &b->ev_t[0], &b->ev_t[1], &b->ev_t[2],
                           &b->ev_t[3], &b->ev_t[4], &b->ev_t[5]})
        if (*e) { cudaEventDestroy(*e); *e = nullptr; }
}

nr_batch* new_batch(const nr_scoring_t* sc, BatchKind kind) {
    if (check_scoring(sc)) return nullptr;
    if (ensure_init(-1)) return nullptr;
    nr_batch* b = new (std::nothrow) nr_batch();
    if (!b) { fail(NR_ERR_NOMEM, "out of host memory"); return nullptr; }
    if (cudaEventCreateWithFlags(&b->ev_uploaded, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&b->ev_done, cudaEventDisableTiming) != cudaSuccess) {
        fail(NR_ERR_CUDA, "cudaEventCreate failed");
        free_events(b);
        delete b;
        return nullptr;
    }
    b->kind = kind;
    b->sc = *sc;
    // the shared-sweep ladder kernels exist for the reference's scoring only (tk.py:502-517: every preset is map-ont);
    // any other scoring scores every rung as its own rectangle (mode 0), which the 32-bit exact kernel does for any values
    const int mode = is_map_ont(*sc) ? g_ladder_mode.load() : 0;
    b->ladder = kind == KIND_ROUND3 && mode != 0;
    b->flag = kind == KIND_ROUND3 && mode >= 2;
    b->pair = kind == KIND_ROUND3 && mode == 3;
    return b;
}

// Paired round 3, long reads: a read whose selection hinges on a tie between a marked and an unmarked candidate (the
// 16-bit words carry no coordinates to order them) is rescored on 32-bit flag words.  For reads of one stripe the device
// does that itself (redo launch); for the stripes of long reads the scratch would have to exist up front for every long
// read, so the (rare: none in any of the five configs' data) cases come back as a list and are rescored here: a batch of
// their own over the same packed reads and templates, the 32-bit ladder, results merged into this batch's records.
int redo_long_reads(nr_batch* b) {
    const int cnt = b->h_redo_count[1];
    std::vector<int32_t> tids((size_t)cnt);
    cudaStream_t st = b->run_stream ? b->run_stream : g_ctx.stream;
    CUDA_TRY(cudaMemcpyAsync(tids.data(), b->d_redo + b->ltasks.size(), sizeof(int32_t) * (size_t)cnt, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    nr_batch* t = new_batch(&b->sc, KIND_ROUND3);
    if (!t) return g_code;
    t->ladder = true; t->flag = true; t->pair = false;          // mode 2 whatever the process-wide ladder mode says
    t->qsrc = b->qsrc;
    if (t->qsrc) ++t->qsrc->refs;
    t->pool.words = b->pool.words;                              // the templates (and the reads, when the batch owns them)
    t->lregs = b->lregs;
    t->regions = b->regions;
    t->rung_off.push_back(0);
    for (int j = 0; j < cnt; ++j) {
        if (tids[j] < 0 || tids[j] >= (int)b->ltasks.size()) { nr_batch_destroy(t); return fail(NR_ERR_CUDA, "corrupt redo list"); }
        nr::LadderTask lt = b->ltasks[tids[j]];
        lt.read = j;
        lt.out_off = (int32_t)t->rung_off.back();
        lt.pad = 0;
        t->ltasks.push_back(lt);
        t->lt_src.push_back(-1);
        t->rung_off.push_back(t->rung_off.back() + (lt.kmax - lt.kmin + 1));
        t->kmin.push_back(lt.kmin); t->kmax.push_back(lt.kmax);
        t->read_region.push_back(0);
    }
    t->n_reads = cnt;
    t->n_out = (size_t)t->rung_off.back();
    int rc = commit_batch(t);
    if (!rc) rc = run_batch(t, st);
    if (!rc) rc = fetch_raw(t);
    if (!rc)
        for (int j = 0; j < cnt; ++j) b->h_sel[b->ltasks[tids[j]].read] = t->h_sel[j];
    nr_batch_destroy(t);
    if (!rc) b->long_redone = true;
    return rc;
}

}  // namespace

// ---- exported C ABI --------------------------------------------------------------------------------------------
extern "C" {

int nr_get_preset(const char* data_type, nr_scoring_t* out) {
    if (!data_type || !out) return fail(NR_ERR_ARG, "nr_get_preset: NULL argument");
    // reference tk.py:502-517: all five data types map to `-x map-ont`
    static const char* names[] = {"ont", "ont_sup", "ont_q20", "clr", "hifi"};
    for (const char* n : names) {
        if (strcmp(n, data_type) == 0) {
            nr_scoring_t s = {2, 4, 4, 2, 24, 1, 1, 80};
            *out = s;
            return NR_OK;
        }
    }
    return fail(NR_ERR_UNKNOWN_TYPE, "Unknown data type: %s", data_type);
}

int nr_init(int device) { return ensure_init(device); }

int nr_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    if (g_ctx.ready) {
        trim_cache_locked();
        cudaStreamDestroy(g_ctx.stream);
        g_ctx = Context();
    }
    return NR_OK;
}

const char* nr_last_error(void) { return g_err.c_str(); }

int nr_device_info(int32_t* device, int32_t* sm_count, int32_t* clock_khz) {
    int rc = ensure_init(-1);
    if (rc) return rc;
    if (device) *device = g_ctx.device;
    if (sm_count) *sm_count = g_ctx.sm_count;
    if (clock_khz) *clock_khz = g_ctx.clock_khz;
    return NR_OK;
}

int nr_set_ladder_mode(int mode) {
    if (mode < 0 || mode > 3) return fail(NR_ERR_ARG, "nr_set_ladder_mode: mode must be 0, 1, 2 or 3");
    g_ladder_mode.store(mode);
    return NR_OK;
}

int nr_limits(int32_t* max_score, int32_t* max_tlen) {
    if (max_score) *max_score = kMaxScore;
    if (max_tlen) *max_tlen = kMaxTlen;
    return NR_OK;
}

void nr_batch_destroy(nr_batch_t* b) {
    if (!b) return;
    if (--b->refs > 0) return;           // a round-3 batch still reads this batch's packed reads: freed with it
    if (b->committed && b->ev_uploaded) cudaEventSynchronize(b->ev_uploaded);   // buffers return to the cache: the upload
    // ... and the kernels and result copies must be done: this batch's own (its event), not whatever another thread's
    // call has queued behind them on the same stream
    if (b->ran && b->ev_done) cudaEventSynchronize(b->ev_done);
    else if (b->ran && b->run_stream) cudaStreamSynchronize(b->run_stream);
    cached_free(b->d_blob, b->blob_bytes, BUF_DEV);
    cached_free(b->h_blob, b->blob_bytes, BUF_PIN);
    cached_free(b->d_out, b->out_bytes, BUF_DEV);
    cached_free(b->h_out, b->out_bytes, BUF_PIN);
    cached_free(b->d_scratch, b->scratch_bytes, BUF_SCRATCH);
    cached_free(b->d_flags, b->flags_bytes, BUF_DEV);
    cached_free(b->d_state, b->state_bytes, BUF_DEV);
    if (b->d_kept) cached_free(b->d_kept, sizeof(uint32_t) * 128 * kWarpsPerBlock * (size_t)g_ctx.sm_count, BUF_DEV);
    cached_free(b->d_sel, b->sel_bytes, BUF_DEV);
    cached_free(b->h_sel, b->sel_bytes, BUF_PIN);
    cached_free(b->d_prung, b->prung_bytes, BUF_DEV);
    cached_free(b->d_redo, b->redo_bytes, BUF_DEV);
    cached_free(b->h_redo_count, 64, BUF_PIN);
    cached_free(b->h_spin, 64, BUF_PIN);
    nr_batch* src = b->qsrc;
    free_events(b);
    delete b;
    if (src) nr_batch_destroy(src);
}

nr_batch_t* nr_batch_begin_round3_from(nr_batch_t* round2) {
    if (!round2 || round2->kind != KIND_ROUND2 || !round2->committed) {
        fail(NR_ERR_ARG, "nr_batch_begin_round3_from: needs a committed round-2 batch");
        return nullptr;
    }
    nr_batch* b = new_batch(&round2->sc, KIND_ROUND3);
    if (!b) return nullptr;
    if (!b->ladder) {
        fail(NR_ERR_ARG, "nr_batch_begin_round3_from: needs a ladder mode (nr_set_ladder_mode 1 or 2)");
        free_events(b);
        delete b;
        return nullptr;
    }
    b->qsrc = round2;
    ++round2->refs;
    return b;
}

int nr_batch_add_round3_reuse(nr_batch_t* b, int32_t region_index, const char* right, int32_t n_right,
                              const int32_t* kmin, const int32_t* kmax) {
    if (!b || !b->qsrc) return fail(NR_ERR_ARG, "nr_batch_add_round3_reuse: batch was not begun with nr_batch_begin_round3_from");
    const nr_batch* src = b->qsrc;
    if (region_index < 0 || region_index >= (int)src->regions.size())
        return fail(NR_ERR_ARG, "nr_batch_add_round3_reuse: region %d is not in the round-2 batch", region_index);
    const RegionInfo& g = src->regions[region_index];
    ReadSrc none = {nullptr, nullptr, nullptr, nullptr, 0};
    return add_round3(b, g.left.data(), g.n_left, right, n_right, g.motif.data(), g.motif_len, g.n_reads, none, kmin, kmax,
                      src->tasks.data() + g.first_read);
}

nr_batch_t* nr_batch_begin(const nr_scoring_t* sc, int32_t kind) {
    if (kind != NR_KIND_ROUND2 && kind != NR_KIND_ROUND3 && kind != NR_KIND_ROUND2_FLAGS) {
        fail(NR_ERR_ARG, "nr_batch_begin: kind must be NR_KIND_ROUND2, NR_KIND_ROUND2_FLAGS or NR_KIND_ROUND3");
        return nullptr;
    }
    nr_batch* b = new_batch(sc, kind == NR_KIND_ROUND3 ? KIND_ROUND3 : KIND_ROUND2);
    if (b && kind == NR_KIND_ROUND2_FLAGS) b->r2flags = b->pair = true;
    return b;
}

int nr_batch_add_round2(nr_batch_t* b, const char* left, int32_t n_left, const char* motif, int32_t motif_len,
                        int32_t T, int32_t n_reads, const char* cores_concat, const int64_t* core_off) {
    if (n_reads > 0 && (!cores_concat || !core_off)) return fail(NR_ERR_ARG, "nr_batch_add_round2: NULL reads");
    ReadSrc src = {nullptr, nullptr, cores_concat, core_off, 0};
    return add_round2(b, left, n_left, motif, motif_len, T, n_reads, src);
}

// reads as one buffer of n_reads lines separated by '\n' (what "\n".join(cores) gives a Python caller without a second
// pass for the lengths); a buffer with another number of lines is rejected like a bad base (a core held a newline)
int nr_batch_add_round2_lines(nr_batch_t* b, const char* left, int32_t n_left, const char* motif, int32_t motif_len,
                              int32_t T, int32_t n_reads, const char* lines, int64_t lines_len) {
    if (n_reads < 0 || lines_len < 0 || (n_reads > 0 && !lines)) return fail(NR_ERR_ARG, "nr_batch_add_round2_lines: bad arguments");
    std::vector<int64_t> off;      // off[r] = start of line r, off[n_reads] = one past the last line's (virtual) newline
    if (n_reads > 0) {
        off.reserve((size_t)n_reads + 1);
        int64_t pos = 0;
        for (;;) {
            off.push_back(pos);
            const char* nl = pos < lines_len ? static_cast<const char*>(memchr(lines + pos, '\n', (size_t)(lines_len - pos))) : nullptr;
            if (!nl) break;
            pos = nl - lines + 1;
        }
        off.push_back(lines_len + 1);
        if ((int64_t)off.size() != (int64_t)n_reads + 1)
            return fail(NR_ERR_BAD_BASE, "nr_batch_add_round2_lines: %lld lines for %d reads (a core holds a newline?)",
                        (long long)off.size() - 1, n_reads);
    }
    ReadSrc src = {nullptr, nullptr, lines, off.data(), 1};
    return add_round2(b, left, n_left, motif, motif_len, T, n_reads, src);
}

int nr_batch_add_round3(nr_batch_t* b, const char* left, int32_t n_left, const char* right, int32_t n_right,
                        const char* motif, int32_t motif_len, int32_t n_reads, const char* cores_concat,
                        const int64_t* core_off, const int32_t* kmin, const int32_t* kmax) {
    if (n_reads > 0 && (!cores_concat || !core_off)) return fail(NR_ERR_ARG, "nr_batch_add_round3: NULL reads");
    if (b && b->qsrc) return fail(NR_ERR_ARG, "nr_batch_add_round3: this batch reuses a round-2 batch's reads (nr_batch_add_round3_reuse)");
    ReadSrc src = {nullptr, nullptr, cores_concat, core_off, 0};
    return add_round3(b, left, n_left, right, n_right, motif, motif_len, n_reads, src, kmin, kmax);
}

int nr_batch_commit(nr_batch_t* b) {
    if (!b || b->committed) return fail(NR_ERR_ARG, "nr_batch_commit: NULL or already committed batch");
    return commit_batch(b);
}

nr_batch_t* nr_batch_create_tasks(const nr_scoring_t* sc, int32_t n_tasks, const char* const* queries,
                                  const int32_t* qlen, const char* const* targets, const int32_t* tlen) {
    if (n_tasks < 0 || (n_tasks > 0 && (!queries || !qlen || !targets || !tlen))) {
        fail(NR_ERR_ARG, "nr_batch_create_tasks: bad arguments");
        return nullptr;
    }
    nr_batch* b = new_batch(sc, KIND_TASKS);
    if (!b) return nullptr;
    b->tasks.resize(n_tasks);
    std::unordered_map<const char*, std::pair<int, uint32_t>> seen;   // pointer -> (len, word): callers often
    for (int i = 0; i < n_tasks; ++i) {                                // pass one template for many reads
        nr::Task& t = b->tasks[i];
        t.q_len = qlen[i];
        t.t_len = tlen[i];
        const char* ptrs[2] = {queries[i], targets[i]};
        const int lens[2] = {qlen[i], tlen[i]};
        uint32_t words[2];
        for (int s = 0; s < 2; ++s) {
            auto it = seen.find(ptrs[s]);
            if (it != seen.end() && it->second.first == lens[s]) { words[s] = it->second.second; continue; }
            const int rc = add_seq(b, ptrs[s], lens[s], s ? "target" : "query", i, &words[s], /*ambiguous_ok=*/s == 0);
            if (rc == NR_ERR_BAD_BASE && s == 1) { words[1] = 0; t.t_len = -1; continue; }     // not scored, record (0, 0, 0)
            if (rc) { nr_batch_destroy(b); return nullptr; }
            seen[ptrs[s]] = std::make_pair(lens[s], words[s]);
        }
        t.q_word = words[0];
        t.t_word = words[1];
    }
    if (commit_batch(b)) { nr_batch_destroy(b); return nullptr; }
    return b;
}

nr_batch_t* nr_batch_create_round2(const nr_scoring_t* sc, const char* left, int32_t n_left, const char* motif,
                                   int32_t motif_len, int32_t T, int32_t n_reads, const char* const* cores,
                                   const int32_t* core_len) {
    if (n_reads > 0 && (!cores || !core_len)) { fail(NR_ERR_ARG, "nr_batch_create_round2: NULL reads"); return nullptr; }
    nr_batch* b = new_batch(sc, KIND_ROUND2);
    if (!b) return nullptr;
    ReadSrc src = {cores, core_len, nullptr, nullptr, 0};
    if (add_round2(b, left, n_left, motif, motif_len, T, n_reads, src) || commit_batch(b)) { nr_batch_destroy(b); return nullptr; }
    return b;
}

nr_batch_t* nr_batch_create_round3(const nr_scoring_t* sc, const char* left, int32_t n_left, const char* right,
                                   int32_t n_right, const char* motif, int32_t motif_len, int32_t n_reads,
                                   const char* const* cores, const int32_t* core_len, const int32_t* kmin,
                                   const int32_t* kmax) {
    if (n_reads > 0 && (!cores || !core_len)) { fail(NR_ERR_ARG, "nr_batch_create_round3: NULL reads"); return nullptr; }
    nr_batch* b = new_batch(sc, KIND_ROUND3);
    if (!b) return nullptr;
    ReadSrc src = {cores, core_len, nullptr, nullptr, 0};
    if (add_round3(b, left, n_left, right, n_right, motif, motif_len, n_reads, src, kmin, kmax) || commit_batch(b)) {
        nr_batch_destroy(b);
        return nullptr;
    }
    return b;
}

int nr_batch_run(nr_batch_t* b, void* stream) {
    if (!b) return fail(NR_ERR_ARG, "nr_batch_run: NULL batch");
    return run_batch(b, stream ? (cudaStream_t)stream : g_ctx.stream);
}

int nr_batch_fetch_alns(nr_batch_t* b, nr_aln_t* out) {
    if (!b || (!out && b->n_out)) return fail(NR_ERR_ARG, "nr_batch_fetch_alns: NULL argument");
    if (b->flag) return fail(NR_ERR_ARG, "nr_batch_fetch_alns: a flag-ladder batch has no (tstart, tend) records; use nr_batch_fetch_round3 or nr_set_ladder_mode(1)");
    if (b->r2flags) return fail(NR_ERR_ARG, "nr_batch_fetch_alns: a NR_KIND_ROUND2_FLAGS batch has no tstart; use nr_batch_fetch_round2");
    int rc = fetch_raw(b);
    if (rc) return rc;
    for (size_t i = 0; i < b->n_out; ++i) {
        out[i].score = b->h_out[i].x;
        out[i].tstart = b->h_out[i].y;
        out[i].tend = b->h_out[i].z;
    }
    return NR_OK;
}

int nr_batch_fetch_round2(nr_batch_t* b, int32_t* score, int32_t* tend, uint8_t* starts_by_left) {
    if (!b || b->kind != KIND_ROUND2) return fail(NR_ERR_ARG, "nr_batch_fetch_round2: not a round-2 batch");
    if (b->n_out && (!score || !tend || !starts_by_left)) return fail(NR_ERR_ARG, "nr_batch_fetch_round2: NULL output");
    int rc = fetch_raw(b);
    if (rc) return rc;
    for (const RegionInfo& g : b->regions)
        for (int r = g.first_read; r < g.first_read + g.n_reads; ++r) {
            const int4 a = b->h_out[r];
            score[r] = a.x;
            tend[r] = a.z;
            starts_by_left[r] = a.y <= g.n_left;      // tstart <= |left| (nanoRepeat_bam.py:373); paired records hold 0 or |left| + 1
        }
    return NR_OK;
}

int nr_batch_fetch_round3(nr_batch_t* b, const int64_t* rung_offset, nr_rung_t* rungs, int64_t* sum_k,
                          int32_t* n_k, int32_t* top_score) {
    if (!b || b->kind != KIND_ROUND3) return fail(NR_ERR_ARG, "nr_batch_fetch_round3: not a round-3 batch");
    if (b->n_reads > 0 && (!sum_k || !n_k || !top_score)) return fail(NR_ERR_ARG, "nr_batch_fetch_round3: NULL output");
    if (rungs && !rung_offset) return fail(NR_ERR_ARG, "rungs given without rung_offset");
    if (rungs && b->pair) return fail(NR_ERR_ARG, "nr_batch_fetch_round3: the paired ladder (mode 3) keeps no rung records; use nr_set_ladder_mode(2)");
    if (b->flag) {
        // the kernel selected per read (nr_kernels.cuh, Sweep::select_rung); the rung records cross the bus only on request
        int rc0 = fetch_raw(b);
        if (rc0) return rc0;
        if (rungs && b->n_out) {
            cudaStream_t st = b->run_stream ? b->run_stream : g_ctx.stream;
            CUDA_TRY(cudaMemcpyAsync(b->h_out, b->d_out, sizeof(int4) * b->n_out, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        for (int r = 0; r < b->n_reads; ++r) {
            const int4 v = b->h_sel[r];
            top_score[r] = v.x;
            n_k[r] = v.y;
            sum_k[r] = (int64_t)(((uint64_t)(uint32_t)v.w << 32) | (uint32_t)v.z);
        }
        if (rungs) {
            for (int r = 0; r < b->n_reads; ++r) {
                const int64_t o = b->rung_off[r];
                const int n = (int)(b->rung_off[r + 1] - o);
                for (int i = 0; i < n; ++i) {
                    const int4 a = b->h_out[o + i];
                    nr_rung_t& rg = rungs[rung_offset[r] + i];
                    rg.score = a.x;
                    rg.starts_in_left = a.y != 0;
                    rg.ends_in_right = a.z != 0;
                    rg.pad[0] = rg.pad[1] = 0;
                }
            }
        }
        b->stats.d2h_bytes = (int64_t)sizeof(int4) * (b->n_reads + (rungs ? (int64_t)b->n_out : 0));
        return NR_OK;
    }
    int rc = fetch_raw(b);
    if (rc) return rc;
    const int min_score = std::max(1, b->sc.min_dp_score);
    for (int r = 0; r < b->n_reads; ++r) {
        const RegionInfo& g = b->regions[b->read_region[r]];
        const int64_t o = b->rung_off[r];
        const int n = (int)(b->rung_off[r + 1] - o);
        int top = 0;
        for (int i = 0; i < n; ++i) {
            int s = b->h_out[o + i].x;
            if (s >= min_score && s > top) top = s;
        }
        int64_t sum = 0;
        int cnt = 0;
        for (int i = 0; i < n; ++i) {
            const int4 a = b->h_out[o + i];
            const int k = b->kmin[r] + i;
            const int tlen = g.n_left + g.motif_len * k + g.n_right;
            const bool in_right = a.x > 0 && tlen - a.z < g.n_right;     // tlen - tend < |right|  (:427)
            const bool in_left = in_right && a.y < g.n_left;             // tstart < |left|; reported only with in_right
            if (rungs) {
                nr_rung_t& rg = rungs[rung_offset[r] + i];
                rg.score = a.x;
                rg.starts_in_left = in_left;
                rg.ends_in_right = in_right;
                rg.pad[0] = rg.pad[1] = 0;
            }
            if (top > 0 && a.x == top && in_left) { sum += k; ++cnt; }
        }
        sum_k[r] = sum;
        n_k[r] = cnt;
        top_score[r] = top;
    }
    return NR_OK;
}

int nr_set_timing(int on) {
    g_timing.store(on ? 1 : 0);
    return NR_OK;
}

int nr_batch_launch_info(nr_batch_t* b, nr_launch_info_t* out) {
    if (!b || !out) return fail(NR_ERR_ARG, "nr_batch_launch_info: NULL argument");
    if (!b->committed) return fail(NR_ERR_ARG, "nr_batch_launch_info: batch was not committed");
    *out = {};
    out->paired_cells = out->planned_paired_cells = b->paired_cells;
    out->rest_cells = b->rest_cells;
    out->paired_useful_cells = out->planned_paired_useful_cells = b->paired_useful;
    out->rest_useful_cells = b->rest_useful;
    out->n_pairs = b->launch.n_pairs;
    out->n_rest = b->launch.count;
    if (b->ran) {
        CUDA_TRY(cudaEventSynchronize(b->ev_done));
        if (b->round2_exit) {       // what the dominance exit skipped in the last run (the counters stay until the next)
            unsigned long long skipped[2];
            CUDA_TRY(cudaMemcpy(skipped, b->d_counters + nr::pr::kExitSlot, sizeof(skipped), cudaMemcpyDeviceToHost));
            out->paired_cells -= 2 * (int64_t)skipped[0];
            out->paired_useful_cells -= (int64_t)(skipped[1] / 32);
        }
        if (b->h_redo_count) out->n_redo = *b->h_redo_count;
        if (b->timed[0]) CUDA_TRY(cudaEventElapsedTime(&out->rest_ms, b->ev_t[0], b->ev_t[1]));
        if (b->timed[1]) CUDA_TRY(cudaEventElapsedTime(&out->paired_ms, b->ev_t[2], b->ev_t[3]));
        if (b->timed[2]) CUDA_TRY(cudaEventElapsedTime(&out->redo_ms, b->ev_t[4], b->ev_t[5]));
    }
    return NR_OK;
}

int nr_batch_stats(const nr_batch_t* b, nr_stats_t* out) {
    if (!b || !out) return fail(NR_ERR_ARG, "nr_batch_stats: NULL argument");
    *out = b->stats;
    return NR_OK;
}

int nr_last_stats(nr_stats_t* out) {
    if (!out) return fail(NR_ERR_ARG, "nr_last_stats: NULL argument");
    *out = g_last_stats;
    return NR_OK;
}

int nr_score_tasks(const nr_scoring_t* sc, int32_t n_tasks, const char* const* queries, const int32_t* qlen,
                   const char* const* targets, const int32_t* tlen, nr_aln_t* out) {
    if (n_tasks > 0 && !out) return fail(NR_ERR_ARG, "nr_score_tasks: out is NULL");
    nr_batch_t* b = nr_batch_create_tasks(sc, n_tasks, queries, qlen, targets, tlen);
    if (!b) return g_code;
    int rc = nr_batch_run(b, nullptr);
    if (!rc) rc = nr_batch_fetch_alns(b, out);
    g_last_stats = b->stats;
    nr_batch_destroy(b);
    return rc;
}

int nr_round2_region(const nr_scoring_t* sc, const char* left, int32_t n_left, const char* motif,
                     int32_t motif_len, int32_t T, int32_t n_reads, const char* const* cores,
                     const int32_t* core_len, nr_aln_t* out) {
    if (n_reads > 0 && !out) return fail(NR_ERR_ARG, "nr_round2_region: out is NULL");
    nr_batch_t* b = nr_batch_create_round2(sc, left, n_left, motif, motif_len, T, n_reads, cores, core_len);
    if (!b) return g_code;
    int rc = nr_batch_run(b, nullptr);
    if (!rc) rc = nr_batch_fetch_alns(b, out);
    g_last_stats = b->stats;
    nr_batch_destroy(b);
    return rc;
}

int nr_round3_region(const nr_scoring_t* sc, const char* left, int32_t n_left, const char* right, int32_t n_right,
                     const char* motif, int32_t motif_len, int32_t n_reads, const char* const* cores,
                     const int32_t* core_len, const int32_t* kmin, const int32_t* kmax,
                     const int64_t* rung_offset, nr_rung_t* rungs, int64_t* sum_k, int32_t* n_k,
                     int32_t* top_score) {
    nr_batch_t* b = nr_batch_create_round3(sc, left, n_left, right, n_right, motif, motif_len, n_reads, cores,
                                           core_len, kmin, kmax);
    if (!b) return g_code;
    int rc = nr_batch_run(b, nullptr);
    if (!rc) rc = nr_batch_fetch_round3(b, rung_offset, rungs, sum_k, n_k, top_score);
    g_last_stats = b->stats;
    nr_batch_destroy(b);
    return rc;
}

}  // extern "C"

// ---- rounds 1-3 of any number of regions in one call --------------------------------------------------------------
// The arithmetic that decides results is the reference's, in IEEE doubles exactly as Python evaluates it (a Python float
// IS a C double; int() truncates toward zero like the casts below; no expression here can be contracted into an FMA):
//   r1 = float(dist) / len(motif); T = int(max r1 * 1.5) + 1, raised to int(max r1 + 10)       nanoRepeat_bam.py:339-347
//   r2 = float(tend - |left|) / len(motif) where tstart <= |left| <= tend                      :373-375
//   buffer = max(15, int(r2 * 0.05)) <= 150 (fast mode: 15); k = int(r2 - buffer) .. int(r2 + buffer), kmin >= 0   :463-472
//   r3 = mean of the tied top rungs that span both anchors (sum and count are exact integers, one division), else r2   :423-433
namespace {

struct Group {
    int r0, r1;
    nr_batch* b2 = nullptr;
    nr_batch* b3 = nullptr;
    std::vector<int> regs;
    int rc = NR_OK;            // of the thread that packed this group's reads
    std::string err;
};

// host threads this process may use (one process per GPU shares the cores with its siblings)
int host_threads() {
    static const int share = [] { const char* e = getenv("LOCAL_WORLD_SIZE"); return e && atoi(e) > 0 ? atoi(e) : 1; }();
    return (int)std::max(1u, std::thread::hardware_concurrency() / (unsigned)share);
}

int estimate_regions(const nr_scoring_t* sc, int fast_mode, int n_regions, const nr_region_t* regs, double* r1, double* r2,
                     uint8_t* r2_valid, double* r3, uint8_t* r3_state, int32_t* T_out, nr_stats_t* stats) {
    std::vector<long long> first(n_regions + 1, 0);
    for (int g = 0; g < n_regions; ++g) {
        const nr_region_t& R = regs[g];
        if (R.n_reads < 0 || R.motif_len <= 0 || !R.motif || (R.n_reads > 0 && (!R.reads || !R.dist_between_anchors)))
            return fail(NR_ERR_ARG, "nr_estimate_regions: region %d has bad arguments", g);
        first[g + 1] = first[g] + R.n_reads;
    }
    const long long total = first[n_regions];
    for (long long i = 0; i < total; ++i) { r2_valid[i] = 0; r3_state[i] = 0; r2[i] = 0.0; r3[i] = 0.0; }
    // ---- round 1 (host): r1 per read, T per region ----
    std::vector<int32_t> T(n_regions, 0);
    for (int g = 0; g < n_regions; ++g) {
        const nr_region_t& R = regs[g];
        if (R.n_reads == 0) continue;                                                   // :336
        const double m = (double)R.motif_len;
        double mx = 0.0;
        for (int r = 0; r < R.n_reads; ++r) {
            const double v = (double)R.dist_between_anchors[r] / m;                     // :341
            r1[first[g] + r] = v;
            if (r == 0 || v > mx) mx = v;
        }
        if (R.has_round1_max_dist) { const double v = (double)R.round1_max_dist / m; if (v > mx) mx = v; }
        int t = (int)(mx * 1.5) + 1;                                                    // :344
        if ((double)t < mx + 10.0) t = (int)(mx + 10.0);                                // :346-347
        if (t < 0) t = 0;
        T[g] = t;
        if (T_out) T_out[g] = t;
    }
    // ---- groups of regions, software-pipelined: while the GPU scores one group the host packs the next ----
    // Short reads: groups of >= 4096 reads, so that packing / planning / selection of one group hide behind the kernels
    // of another.  Long reads (cores of a kilobase and more on average) are the opposite case: the host work is
    // negligible beside the kernels, and every launch pays the serial chain of its longest read's stripes once, so the
    // whole call is one group.
    // (measured on the 60 000-read slice of config 3: groups of 16 384 reads 49 ms end to end, of 4 096 reads 63 ms --
    // a launch of 2 500 pairs on 2 368 warp slots takes as long as one of 4 700; on config 2's 10 000 reads two groups of
    // 5 000 beat one of 10 000 by 0.3 ms)
    long long kMinReads = total >= 12288 ? 16384 : 4096;
    if (const char* e = getenv("NR_GROUP_READS")) kMinReads = std::max(256, atoi(e));      // tuning
    long long total_bases = 0;
    for (int g = 0; g < n_regions; ++g) total_bases += regs[g].reads_len;
    const bool long_reads = total > 0 && total_bases / total > 1000;
    const int n_groups = long_reads ? 1 : (int)std::max<long long>(1, std::min<long long>(8, total / kMinReads));
    std::vector<Group> groups;
    {
        const double target = (double)total / n_groups;
        long long acc = 0;
        int start = 0;
        for (int g = 0; g < n_regions; ++g) {
            acc += regs[g].n_reads;
            if (acc >= target * (double)(groups.size() + 1) && (int)groups.size() < n_groups - 1) {
                Group G; G.r0 = start; G.r1 = g + 1; groups.push_back(G);
                start = g + 1;
            }
        }
        Group G; G.r0 = start; G.r1 = n_regions; groups.push_back(G);
    }
    int rc = NR_OK;
    auto cleanup = [&]() { for (Group& G : groups) { if (G.b3) nr_batch_destroy(G.b3); if (G.b2) nr_batch_destroy(G.b2); G.b2 = G.b3 = nullptr; } };
    auto add_stats = [&](const nr_batch* b) {
        if (!stats) return;
        stats->algorithmic_cells += b->stats.algorithmic_cells; stats->executed_cells += b->stats.executed_cells;
        stats->n_tasks += b->stats.n_tasks; stats->kernel_launches += b->stats.kernel_launches;
        stats->n_skipped += b->stats.n_skipped; stats->h2d_bytes += b->stats.h2d_bytes; stats->d2h_bytes += b->stats.d2h_bytes;
    };
    if (stats) *stats = {};
    const int min_score = std::max(1, sc->min_dp_score);
    PhaseTrace trace;
    trace.mark("estimate: round 1, grouping");
    // round 2 of every group (was pymm2.main at :362).  The reads of the groups are packed side by side on host threads
    // (pure CPU work on each group's own batch; batches are created here, on the thread that owns the CUDA context),
    // then committed and launched back to back.
    for (Group& G : groups) {
        long long bases = 0;
        for (int g = G.r0; g < G.r1; ++g)
            if (regs[g].n_reads > 0) { G.regs.push_back(g); bases += regs[g].reads_len + regs[g].n_left + (long long)regs[g].motif_len * T[g]; }
        if (G.regs.empty()) continue;
        if (!(G.b2 = nr_batch_begin(sc, NR_KIND_ROUND2_FLAGS))) { cleanup(); return g_code; }
        G.b2->pool.words.reserve((size_t)(bases / 16 + 2 * (long long)G.regs.size() + 64));
        long long n_reads = 0;
        for (int g : G.regs) n_reads += regs[g].n_reads;
        G.b2->pool.words.reserve((size_t)(bases / 16 + 2 * n_reads + 4 * (long long)G.regs.size() + 64));
        G.b2->tasks.reserve((size_t)n_reads);
    }
    static const long long kPackJobReads = [] { const char* e = getenv("NR_PACK_JOB_READS"); return e && atoi(e) > 0 ? (long long)atoi(e) : 4096LL; }();
    // Packing jobs: a group's regions in runs of about 4 096 reads, each run packed by one host thread into a batch of
    // its own (no CUDA objects), the runs then appended to the group's batch in order (word indices shifted).
    struct Job { Group* G; size_t i0, i1; std::unique_ptr<nr_batch> part; int rc = NR_OK; std::string err; };
    std::vector<Job> jobs;
    {
        const int nt_all = host_threads();
        for (Group& G : groups) {
            if (!G.b2) continue;
            long long n_reads = 0;
            for (int g : G.regs) n_reads += regs[g].n_reads;
            const int parts = (int)std::max<long long>(1, std::min<long long>(std::min<long long>(nt_all, 16), n_reads / kPackJobReads));
            const double per = (double)n_reads / parts;
            long long acc = 0;
            size_t start = 0;
            int made = 0;
            for (size_t i = 0; i < G.regs.size(); ++i) {
                acc += regs[G.regs[i]].n_reads;
                if (made < parts - 1 && acc >= per * (made + 1)) { jobs.push_back({&G, start, i + 1, nullptr}); start = i + 1; ++made; }
            }
            if (start < G.regs.size()) jobs.push_back({&G, start, G.regs.size(), nullptr});
        }
        auto pack_job = [&](Job& J) {
            J.part.reset(new (std::nothrow) nr_batch());
            if (!J.part) { J.rc = NR_ERR_NOMEM; J.err = "out of host memory"; return; }
            nr_batch* pb = J.part.get();
            pb->kind = KIND_ROUND2;
            pb->sc = *sc;
            long long bases = 0, n_reads = 0;
            for (size_t i = J.i0; i < J.i1; ++i) {
                const nr_region_t& R = regs[J.G->regs[i]];
                bases += R.reads_len + R.n_left + (long long)R.motif_len * T[J.G->regs[i]];
                n_reads += R.n_reads;
            }
            pb->pool.words.reserve((size_t)(bases / 16 + 2 * n_reads + 4 * (long long)(J.i1 - J.i0) + 64));
            pb->tasks.reserve((size_t)n_reads);
            for (size_t i = J.i0; i < J.i1; ++i) {
                const int g = J.G->regs[i];
                const nr_region_t& R = regs[g];
                const int rc1 = nr_batch_add_round2_lines(pb, R.left, R.n_left, R.motif, R.motif_len, T[g], R.n_reads, R.reads, R.reads_len);
                if (rc1) { J.rc = rc1; J.err = g_err; return; }      // (the message lives in this thread's g_err)
            }
        };
        const int nt = std::min<int>((int)jobs.size(), nt_all);
        if (nt <= 1) {
            for (Job& J : jobs) pack_job(J);
        } else {
            std::atomic<int> next{0};
            auto work = [&]() { for (int i; (i = next.fetch_add(1)) < (int)jobs.size();) pack_job(jobs[i]); };
            std::vector<std::thread> th;
            for (int t = 1; t < nt; ++t) th.emplace_back(work);
            work();
            for (auto& x : th) x.join();
        }
        for (Job& J : jobs) {
            Group& G = *J.G;
            if (G.rc) continue;
            if (J.rc) { G.rc = J.rc; G.err = J.err; continue; }
            nr_batch* pb = J.part.get();
            nr_batch* b = G.b2;
            const size_t base_w = b->pool.words.size();
            if (base_w + pb->pool.words.size() > 0xfffffff0ULL) { G.rc = NR_ERR_TOO_LARGE; G.err = "sequence pool exceeds 2^32 words"; continue; }
            b->pool.words.insert(b->pool.words.end(), pb->pool.words.begin(), pb->pool.words.end());
            const size_t base_t = b->tasks.size();
            b->tasks.insert(b->tasks.end(), pb->tasks.begin(), pb->tasks.end());
            for (size_t t = base_t; t < b->tasks.size(); ++t) { b->tasks[t].q_word += (uint32_t)base_w; b->tasks[t].t_word += (uint32_t)base_w; }
            for (RegionInfo& ri : pb->regions) { ri.first_read += b->n_reads; b->regions.push_back(std::move(ri)); }
            b->n_reads += pb->n_reads;
            b->n_ambiguous_reads += pb->n_ambiguous_reads;
            J.part.reset();
        }
    }
    trace.mark("estimate: round-2 add (pack, threads)");
    for (Group& G : groups) {
        if (G.rc) { const int rc1 = G.rc; const std::string msg = G.err; cleanup(); return fail(rc1, "%s", msg.c_str()); }
        if (G.b2 && ((rc = nr_batch_commit(G.b2)) || (rc = nr_batch_run(G.b2, aux_stream_for(G.b2))))) { cleanup(); return rc; }
        trace.mark("estimate: round-2 commit + run");
    }
    // round-2 selection and the launch of round 3 (was pymm2.main per read at :497), group by group
    std::vector<int32_t> kmin, kmax;
    for (Group& G : groups) {
        if (!G.b2) continue;
        if ((rc = fetch_raw(G.b2))) { cleanup(); return rc; }
        trace.mark("estimate: wait for round 2");
        if (!(G.b3 = nr_batch_begin_round3_from(G.b2))) { cleanup(); return g_code; }
        for (size_t i = 0; i < G.regs.size(); ++i) {
            const int g = G.regs[i];
            const nr_region_t& R = regs[g];
            const RegionInfo& info = G.b2->regions[i];
            const double m = (double)R.motif_len;
            kmin.assign(R.n_reads, 0);
            kmax.assign(R.n_reads, -1);
            for (int r = 0; r < R.n_reads; ++r) {
                const int4 a = G.b2->h_out[info.first_read + r];          // (score, 0 or |left| + 1, tend)
                if (a.x < min_score || a.y > R.n_left || a.z < R.n_left) continue;      // no PAF line below -s; span test :373
                const double v = (double)(a.z - R.n_left) / m;                           // :375
                r2[first[g] + r] = v;
                r2_valid[first[g] + r] = 1;
                int buffer = std::max(15, (int)(v * 0.05));                              // :463-467
                if (buffer > 150) buffer = 150;
                if (fast_mode) buffer = 15;
                kmax[r] = (int)(v + (double)buffer);                                     // :469-472
                kmin[r] = std::max((int)(v - (double)buffer), 0);
            }
            if ((rc = nr_batch_add_round3_reuse(G.b3, (int)i, R.right, R.n_right, kmin.data(), kmax.data()))) { cleanup(); return rc; }
        }
        trace.mark("estimate: select 2 + round-3 add");
        if ((rc = nr_batch_commit(G.b3)) || (rc = nr_batch_run(G.b3, aux_stream_for(G.b3)))) { cleanup(); return rc; }
        trace.mark("estimate: round-3 commit + run");
    }
    // round-3 selection (:423-433)
    for (Group& G : groups) {
        if (!G.b3) continue;
        if ((rc = fetch_raw(G.b3))) { cleanup(); return rc; }
        trace.mark("estimate: wait for round 3");
        for (size_t i = 0; i < G.regs.size(); ++i) {
            const int g = G.regs[i];
            const RegionInfo& info = G.b3->regions[i];
            for (int r = 0; r < regs[g].n_reads; ++r) {
                const long long o = first[g] + r;
                if (!r2_valid[o]) continue;                                              // :460
                const int4 v = G.b3->h_sel[info.first_read + r];                         // (top, n tied, sum k lo, hi)
                if (v.x <= 0) continue;                                                  // no PAF line at all (:421)
                if (v.y > 0) {
                    const long long sum = (long long)(((unsigned long long)(unsigned)v.w << 32) | (unsigned)v.z);
                    r3[o] = (double)sum / (double)v.y;                                   // np.mean of the tied k (:431)
                    r3_state[o] = 1;
                } else {
                    r3[o] = r2[o];                                                       // :433
                    r3_state[o] = 2;
                }
            }
        }
        add_stats(G.b2);
        add_stats(G.b3);
    }
    trace.mark("estimate: select 3");
    cleanup();
    trace.mark("estimate: destroy batches");
    return NR_OK;
}

}  // namespace

extern "C" int nr_estimate_regions(const nr_scoring_t* sc, int32_t fast_mode, int32_t n_regions, const nr_region_t* regions,
                                   double* r1, double* r2, uint8_t* r2_valid, double* r3, uint8_t* r3_state, int32_t* T_out,
                                   nr_stats_t* stats) {
    if (check_scoring(sc)) return g_code;
    if (n_regions < 0 || (n_regions > 0 && !regions)) return fail(NR_ERR_ARG, "nr_estimate_regions: bad arguments");
    long long total = 0;
    for (int g = 0; g < n_regions; ++g) total += std::max(0, regions[g].n_reads);
    if (total > 0 && (!r1 || !r2 || !r2_valid || !r3 || !r3_state)) return fail(NR_ERR_ARG, "nr_estimate_regions: NULL output");
    if (!is_map_ont(*sc) || g_ladder_mode.load() == 0)
        return fail(NR_ERR_ARG, "nr_estimate_regions needs map-ont scoring and a shared-sweep ladder mode (1-3)");
    return estimate_regions(sc, fast_mode, n_regions, regions, r1, r2, r2_valid, r3, r3_state, T_out, stats);
}

// ---- what the other host translation units (nr_joint.cu, nr_anchor.cu) share with this one ----------------------------
namespace nri {
int ensure_init() { return ::ensure_init(-1); }
cudaStream_t stream() { return g_ctx.stream; }
int sm_count() { return g_ctx.sm_count; }
int fail_msg(int code, const char* msg) { return fail(code, "%s", msg); }
int last_code() { return g_code; }
bool pack(const char* s, int len, uint32_t* w) { return pack_seq(s, len, w); }
void ambiguity(const char* s, int len, uint32_t* m) { ambiguity_plane(s, len, m); }
int alloc(void** p, size_t bytes, bool pinned) { return cached_alloc(p, bytes, pinned ? BUF_PIN : BUF_DEV); }
void release(void* p, size_t bytes, bool pinned) { cached_free(p, bytes, pinned ? BUF_PIN : BUF_DEV); }
int check(const nr_scoring_t* sc) { return check_scoring(sc); }
}  // namespace nri
