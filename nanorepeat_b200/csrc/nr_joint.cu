// nr_joint.cu -- host side + launcher of the joint path (nanoRepeat-joint): alignment score and window score of every
// (read, template) task in one DP (nr_window_kernel.cuh).  C ABI: nr_window_tasks, nr_joint_grid.
#include "nr_internal.h"
#include "nr_window_kernel.cuh"
#include "nr_window_ladder.cuh"

#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <mutex>
#include <string>
#include <vector>

namespace {

#define JTRY(expr)                                                                                       \
    do {                                                                                                 \
        cudaError_t e__ = (expr);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            char b__[256];                                                                               \
            snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return nri::fail_msg(NR_ERR_CUDA, b__);                                                      \
        }                                                                                                \
    } while (0)

struct SeqPool {
    std::vector<uint32_t> words;
    // read: bases other than ACGT get an ambiguity plane (linked from the slack word); template: must be ACGT (-1)
    long long add(const char* s, int len, bool is_read) {
        const size_t w0 = words.size();
        words.resize(w0 + (size_t)(len + 15) / 16 + 1, 0u);
        if (!nri::pack(s, len, words.data() + w0)) {
            if (!is_read) { words.resize(w0); return -1; }
            const size_t at = words.size();
            words.resize(at + (size_t)(len + 31) / 32, 0u);
            nri::ambiguity(s, len, words.data() + at);
            words[w0 + (size_t)(len + 15) / 16] = (uint32_t)(at - w0);
        }
        return (long long)w0;
    }
};

// The joint path's limits (include/nanorepeat_b200.h): the DP word holds score * 65536 + payload, so the score must stay
// within 15 bits and the window within 8 000 bases (payload <= +16 000); the per-warp scratch row holds one template.
constexpr int kMaxScore = 32767, kMaxWindow = 8000, kMaxTlen = 1 << 20;

// Every pool word a kernel reads through a 32-bit task field must fit it.
int check_pool(const SeqPool& pool, const char* who) {
    if (pool.words.size() + 4 > (size_t)UINT32_MAX) return nri::fail_msg(NR_ERR_ARG, who);
    return NR_OK;
}

// tasks[i].q_word / t_word index `pool`; out[i] = (score, window score).  skipped[i] (in: 1 for a template the pool could
// not pack) is set for every task beyond the limits above; a skipped task is not scored and its record stays (0, 0).
int run_window_tasks(const nr_scoring_t* sc, std::vector<nrw::WinTask>& tasks, const SeqPool& pool, nr_window_t* out,
                     std::vector<uint8_t>& skipped, int& launches) {
    const int n = (int)tasks.size();
    if (n == 0) return NR_OK;
    if (int rc = check_pool(pool, "joint path: more than 2^32 words of packed sequence in one call")) return rc;
    int max_t = 1;
    for (int i = 0; i < n; ++i) {
        nrw::WinTask& t = tasks[i];
        const long long m = (long long)sc->match * std::min(t.q_len, t.t_len);
        if (m > kMaxScore || t.win_b - t.win_a > kMaxWindow || t.t_len > kMaxTlen) { t.q_len = 0; skipped[i] = 1; }
        max_t = std::max(max_t, t.t_len);
    }
    // long tasks first: the tail of the launch is made of short ones
    std::vector<int> order(n);
    for (int i = 0; i < n; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int x, int y) {
        const long long cx = (long long)tasks[x].q_len * tasks[x].t_len, cy = (long long)tasks[y].q_len * tasks[y].t_len;
        return cx != cy ? cx > cy : x < y;
    });
    std::vector<nrw::WinTask> sorted(n);
    for (int i = 0; i < n; ++i) sorted[i] = tasks[order[i]];
    const int blocks = std::max(1, std::min(2 * nri::sm_count(), (n + nrw::kWarps - 1) / nrw::kWarps));
    const int stride = 2 * ((max_t + 31) / 32 * 32);
    const size_t task_bytes = sizeof(nrw::WinTask) * n, pool_bytes = sizeof(uint32_t) * (pool.words.size() + 4),
                 out_bytes = sizeof(int2) * n, scratch_bytes = sizeof(int4) * (size_t)blocks * nrw::kWarps * stride;
    void *d_tasks = nullptr, *d_pool = nullptr, *d_out = nullptr, *d_scratch = nullptr, *d_counter = nullptr, *h_out = nullptr;
    int rc;
    auto cleanup = [&]() {
        nri::release(d_tasks, task_bytes, false); nri::release(d_pool, pool_bytes, false); nri::release(d_out, out_bytes, false);
        nri::release(d_scratch, scratch_bytes, false); nri::release(d_counter, 256, false); nri::release(h_out, out_bytes, true);
    };
    if ((rc = nri::alloc(&d_tasks, task_bytes, false)) || (rc = nri::alloc(&d_pool, pool_bytes, false)) ||
        (rc = nri::alloc(&d_out, out_bytes, false)) || (rc = nri::alloc(&d_scratch, scratch_bytes, false)) ||
        (rc = nri::alloc(&d_counter, 256, false)) || (rc = nri::alloc(&h_out, out_bytes, true))) { cleanup(); return rc; }
    cudaStream_t st = nri::stream();
    nrw::WinScore k;
    k.match = sc->match << 16; k.mismatch = -(sc->mismatch << 16); k.ambiguous = -(sc->ambiguous << 16);
    k.open1 = -((sc->gap_open1 + sc->gap_ext1) << 16); k.ext1 = -(sc->gap_ext1 << 16);
    k.open2 = -((sc->gap_open2 + sc->gap_ext2) << 16); k.ext2 = -(sc->gap_ext2 << 16);
    const size_t smem = (size_t)nrw::kWarps * 8 * nrw::kRows * sizeof(int);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&]() { attr_err = cudaFuncSetAttribute(nrw::window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
    cudaError_t e = attr_err;
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_tasks, sorted.data(), task_bytes, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_pool, pool.words.data(), sizeof(uint32_t) * pool.words.size(), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_counter, 0, 256, st);
    if (e == cudaSuccess) {
        nrw::window_kernel<<<blocks, 32 * nrw::kWarps, smem, st>>>(static_cast<const nrw::WinTask*>(d_tasks), n, static_cast<const uint32_t*>(d_pool), k,
                                                                  static_cast<int4*>(d_scratch), stride, static_cast<int*>(d_counter),
                                                                  static_cast<int2*>(d_out));
        e = cudaGetLastError();
        ++launches;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, st);
    const auto t_launch = std::chrono::steady_clock::now();
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (getenv("NR_TRACE"))
        fprintf(stderr, "[nr trace] window kernel: %d tasks, upload + kernel + download %.1f us\n", n,
                std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_launch).count());
    if (e != cudaSuccess) { cleanup(); cudaGetLastError(); return nri::fail_msg(NR_ERR_CUDA, cudaGetErrorString(e)); }
    const int2* res = static_cast<const int2*>(h_out);
    for (int i = 0; i < n; ++i) { out[order[i]].score = res[i].x; out[order[i]].window_score = res[i].y; }
    cleanup();
    return NR_OK;
}

// Device and pinned buffers of one call, given back to the caching allocator on scope exit.
struct Bufs {
    struct One { void* p; size_t bytes; bool pinned; };
    std::vector<One> all;
    int get(void** p, size_t bytes, bool pinned) {
        *p = nullptr;
        const int rc = nri::alloc(p, bytes, pinned);
        if (rc == NR_OK) all.push_back({*p, bytes, pinned});
        return rc;
    }
    ~Bufs() { for (const One& b : all) nri::release(b.p, b.bytes, b.pinned); }
};

nrw::WinScore window_score_words(const nr_scoring_t* sc) {
    nrw::WinScore k;
    k.match = sc->match << 16; k.mismatch = -(sc->mismatch << 16); k.ambiguous = -(sc->ambiguous << 16);
    k.open1 = -((sc->gap_open1 + sc->gap_ext1) << 16); k.ext1 = -(sc->gap_ext1 << 16);
    k.open2 = -((sc->gap_open2 + sc->gap_ext2) << 16); k.ext2 = -(sc->gap_ext2 << 16);
    return k;
}

// The shared-sweep path (nr_window_ladder.cuh): backward tasks, then forward tasks; res[out_off + j] of every forward task.
int run_ladder_tasks(const nr_scoring_t* sc, const std::vector<nrw::LadBwdTask>& btasks, std::vector<nrw::LadFwdTask>& ptasks,
                     std::vector<nrw::LadFwdTask>& ftasks, const SeqPool& pool, size_t bvec_words, size_t cstate_words, size_t n_pbest1,
                     size_t n_out, int max_t, std::vector<int2>& res, int& launches) {
    const int nb = (int)btasks.size(), nf = (int)ftasks.size(), np = (int)ptasks.size();
    res.assign(n_out, make_int2(0, 0));
    if (nf == 0) return NR_OK;
    // long tasks first
    auto by_cost = [](const nrw::LadFwdTask& x, const nrw::LadFwdTask& y) {
        const long long cx = (long long)x.q_len * (x.n_pre + (long long)x.m2 * (x.k2_first + (long long)x.k2_step * (x.k2_count - 1)));
        const long long cy = (long long)y.q_len * (y.n_pre + (long long)y.m2 * (y.k2_first + (long long)y.k2_step * (y.k2_count - 1)));
        return cx != cy ? cx > cy : x.out_off < y.out_off;
    };
    std::sort(ftasks.begin(), ftasks.end(), by_cost);
    std::sort(ptasks.begin(), ptasks.end(), by_cost);
    const int blocks_b = std::max(1, std::min(2 * nri::sm_count(), (nb + nrw::kWarps - 1) / nrw::kWarps));
    const int blocks_f = std::max(1, std::min(2 * nri::sm_count(), (nf + nrw::kWarps - 1) / nrw::kWarps));
    const int blocks_p = std::max(1, std::min(2 * nri::sm_count(), (np + nrw::kWarps - 1) / nrw::kWarps));
    const int stride = 2 * ((max_t + 31) / 32 * 32);
    const size_t scratch_bytes = sizeof(int4) * (size_t)std::max(std::max(blocks_b, blocks_f), blocks_p) * nrw::kWarps * stride;
    const size_t out_bytes = sizeof(int2) * n_out;
    Bufs bufs;
    void *d_b = nullptr, *d_f = nullptr, *d_p = nullptr, *d_pool = nullptr, *d_out = nullptr, *d_scratch = nullptr, *d_counter = nullptr,
         *d_bvec = nullptr, *d_ronly = nullptr, *d_cstate = nullptr, *d_pbest1 = nullptr, *h_out = nullptr;
    int rc;
    if ((rc = bufs.get(&d_b, sizeof(nrw::LadBwdTask) * nb, false)) || (rc = bufs.get(&d_f, sizeof(nrw::LadFwdTask) * nf, false)) ||
        (rc = bufs.get(&d_p, sizeof(nrw::LadFwdTask) * std::max(np, 1), false)) ||
        (rc = bufs.get(&d_cstate, sizeof(int) * std::max<size_t>(cstate_words, 1), false)) ||
        (rc = bufs.get(&d_pbest1, sizeof(int) * std::max<size_t>(n_pbest1, 1), false)) ||
        (rc = bufs.get(&d_pool, sizeof(uint32_t) * (pool.words.size() + 4), false)) || (rc = bufs.get(&d_out, out_bytes, false)) ||
        (rc = bufs.get(&d_scratch, scratch_bytes, false)) || (rc = bufs.get(&d_counter, 256, false)) ||
        (rc = bufs.get(&d_bvec, sizeof(int) * std::max<size_t>(bvec_words, 1), false)) ||
        (rc = bufs.get(&d_ronly, sizeof(int) * nb, false)) || (rc = bufs.get(&h_out, out_bytes, true)))
        return rc;
    cudaStream_t st = nri::stream();
    const nrw::WinScore k = window_score_words(sc);
    const size_t smem_b = (size_t)nrw::kWarps * 8 * nrw::kRows * sizeof(int);
    const size_t smem_f = (size_t)nrw::kWarps * (11 * nrw::kRows + 2 * nrw::kMaxK2) * sizeof(int);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&]() {
        attr_err = cudaFuncSetAttribute(nrw::ladder_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b);
        if (attr_err == cudaSuccess)
            attr_err = cudaFuncSetAttribute(nrw::ladder_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_f);
    });
    JTRY(attr_err);
    JTRY(cudaMemcpyAsync(d_b, btasks.data(), sizeof(nrw::LadBwdTask) * nb, cudaMemcpyHostToDevice, st));
    JTRY(cudaMemcpyAsync(d_f, ftasks.data(), sizeof(nrw::LadFwdTask) * nf, cudaMemcpyHostToDevice, st));
    if (np) JTRY(cudaMemcpyAsync(d_p, ptasks.data(), sizeof(nrw::LadFwdTask) * np, cudaMemcpyHostToDevice, st));
    JTRY(cudaMemcpyAsync(d_pool, pool.words.data(), sizeof(uint32_t) * pool.words.size(), cudaMemcpyHostToDevice, st));
    JTRY(cudaMemsetAsync(d_counter, 0, 256, st));
    int* counter = static_cast<int*>(d_counter);
    nrw::ladder_bwd_kernel<<<blocks_b, 32 * nrw::kWarps, smem_b, st>>>(static_cast<const nrw::LadBwdTask*>(d_b), nb,
                                                                     static_cast<const uint32_t*>(d_pool), k, static_cast<int4*>(d_scratch),
                                                                     stride, counter, static_cast<int*>(d_bvec), static_cast<int*>(d_ronly));
    JTRY(cudaGetLastError());
    ++launches;
    if (np) {       // prefix sweeps: the columns the continuation sweeps start from
        nrw::ladder_fwd_kernel<<<blocks_p, 32 * nrw::kWarps, smem_f, st>>>(static_cast<const nrw::LadFwdTask*>(d_p), np,
                                                                         static_cast<const nrw::LadBwdTask*>(d_b), static_cast<const uint32_t*>(d_pool),
                                                                         k, static_cast<int4*>(d_scratch), stride, counter + 16,
                                                                         static_cast<const int*>(d_bvec), static_cast<const int*>(d_ronly),
                                                                         static_cast<int*>(d_cstate), static_cast<int*>(d_pbest1),
                                                                         static_cast<int2*>(d_out));
        JTRY(cudaGetLastError());
        ++launches;
    }
    nrw::ladder_fwd_kernel<<<blocks_f, 32 * nrw::kWarps, smem_f, st>>>(static_cast<const nrw::LadFwdTask*>(d_f), nf,
                                                                     static_cast<const nrw::LadBwdTask*>(d_b), static_cast<const uint32_t*>(d_pool),
                                                                     k, static_cast<int4*>(d_scratch), stride, counter + 32,
                                                                     static_cast<const int*>(d_bvec), static_cast<const int*>(d_ronly),
                                                                     static_cast<int*>(d_cstate), static_cast<int*>(d_pbest1),
                                                                     static_cast<int2*>(d_out));
    JTRY(cudaGetLastError());
    ++launches;
    JTRY(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    const auto t_launch = std::chrono::steady_clock::now();
    const cudaError_t e = cudaStreamSynchronize(st);
    if (getenv("NR_TRACE"))
        fprintf(stderr, "[nr trace] joint ladder: %d backward + %d prefix + %d forward tasks, %zu grid points, kernels + download %.1f us\n", nb, np,
                nf, n_out, std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_launch).count());
    if (e != cudaSuccess) { cudaGetLastError(); return nri::fail_msg(NR_ERR_CUDA, cudaGetErrorString(e)); }
    std::copy(static_cast<const int2*>(h_out), static_cast<const int2*>(h_out) + n_out, res.begin());
    return NR_OK;
}

}  // namespace

extern "C" int nr_window_tasks(const nr_scoring_t* sc, int32_t n_tasks, const char* const* queries, const int32_t* qlen,
                               const char* const* targets, const int32_t* tlen, const int32_t* win_a, const int32_t* win_b,
                               const uint8_t* reverse, nr_window_t* out) {
    if (nri::check(sc)) return nri::last_code();
    if (n_tasks < 0 || (n_tasks > 0 && (!queries || !qlen || !targets || !tlen || !win_a || !win_b || !out)))
        return nri::fail_msg(NR_ERR_ARG, "nr_window_tasks: bad arguments");
    int rc = nri::ensure_init();
    if (rc) return rc;
    nr_stats_t st = {};
    st.n_tasks = n_tasks;
    nri::set_last_stats(st);
    SeqPool pool;
    std::vector<nrw::WinTask> tasks(n_tasks);
    std::vector<uint8_t> skipped(n_tasks, 0);
    std::map<std::pair<const char*, int>, long long> seen_q, seen_t;
    for (int i = 0; i < n_tasks; ++i) {
        nrw::WinTask& t = tasks[i];
        t = {};
        out[i].score = out[i].window_score = 0;
        if (qlen[i] < 0 || tlen[i] < 0) return nri::fail_msg(NR_ERR_ARG, "nr_window_tasks: negative length");
        auto qk = std::make_pair(queries[i], (int)qlen[i]);
        auto tk = std::make_pair(targets[i], (int)tlen[i]);
        if (!seen_q.count(qk)) seen_q[qk] = pool.add(queries[i], qlen[i], true);
        if (!seen_t.count(tk)) seen_t[tk] = pool.add(targets[i], tlen[i], false);
        const long long tw = seen_t[tk];
        t.q_word = (uint32_t)seen_q[qk]; t.q_len = qlen[i];
        t.t_word = tw < 0 ? 0u : (uint32_t)tw; t.t_len = tw < 0 ? 0 : tlen[i];      // a template with N is not scored
        skipped[i] = tw < 0;
        t.win_a = std::max(0, win_a[i]); t.win_b = std::min(win_b[i], tlen[i]);
        t.reverse = reverse ? reverse[i] != 0 : 0;
    }
    int launches = 0;
    rc = run_window_tasks(sc, tasks, pool, out, skipped, launches);
    st.kernel_launches = launches;
    for (uint8_t k : skipped) st.n_skipped += k;
    nri::set_last_stats(st);
    return rc;
}

extern "C" int nr_joint_grid(const nr_scoring_t* sc, const char* left, int32_t n_left, const char* mid, int32_t n_mid,
                             const char* right, int32_t n_right, const char* motif1, int32_t m1, const char* motif2, int32_t m2,
                             int32_t n_reads, const char* const* reads, const int32_t* read_len, int32_t n_points,
                             const int32_t* point_read, const int32_t* point_k1, const int32_t* point_k2, nr_window_t* out,
                             uint8_t* strand) {
    if (nri::check(sc)) return nri::last_code();
    if (n_left < 0 || n_mid < 0 || n_right < 0 || m1 <= 0 || m2 <= 0 || n_reads < 0 || n_points < 0 || !motif1 || !motif2 ||
        (n_left > 0 && !left) || (n_mid > 0 && !mid) || (n_right > 0 && !right) || (n_reads > 0 && (!reads || !read_len)) ||
        (n_points > 0 && (!point_read || !point_k1 || !point_k2 || !out)))
        return nri::fail_msg(NR_ERR_ARG, "nr_joint_grid: bad arguments");
    int rc = nri::ensure_init();
    if (rc) return rc;
    nr_stats_t st = {};
    st.n_tasks = n_points;
    nri::set_last_stats(st);
    int launches = 0;
    const bool tracing = getenv("NR_TRACE") != nullptr;
    auto t_mark = std::chrono::steady_clock::now();
    auto mark = [&](const char* what) {
        if (!tracing) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[nr trace] joint grid: %-24s %8.1f us\n", what, std::chrono::duration<double, std::micro>(t1 - t_mark).count());
        t_mark = t1;
    };
    SeqPool pool;
    std::vector<long long> read_word(n_reads);
    {
        size_t words = 0;
        for (int r = 0; r < n_reads; ++r) words += (size_t)(std::max(read_len[r], 0) + 15) / 16 + 2;
        pool.words.reserve(words + 4096);
    }
    for (int r = 0; r < n_reads; ++r) {
        if (read_len[r] < 0) return nri::fail_msg(NR_ERR_ARG, "nr_joint_grid: negative read length");
        read_word[r] = pool.add(reads[r], read_len[r], true);
    }
    mark("pack reads");
    for (int i = 0; i < n_points; ++i) {
        if (point_read[i] < 0 || point_read[i] >= n_reads || point_k1[i] < 0 || point_k2[i] < 0)
            return nri::fail_msg(NR_ERR_ARG, "nr_joint_grid: bad grid point");
        out[i].score = out[i].window_score = 0;
        if (strand) strand[i] = 0;
    }
    const int win_a = std::max(n_left - 10, 0);                                                   // nanoRepeat_joint.py:448-451

    // ---- shared sweeps (nr_window_ladder.cuh) for every read whose points are a full K1 x K2 grid with K2 an arithmetic
    // progression (what joint.py's round-2 and round-3 grids are); everything else is scored template by template below.
    std::vector<char> by_ladder(n_points, 0);
    std::vector<int> point_slot(n_points, -1);                      // record of strand '+'; strand '-' follows at +k2_count ... see below
    std::vector<int> point_slot_rev(n_points, -1);
    std::vector<nrw::LadBwdTask> btasks;
    std::vector<nrw::LadFwdTask> ftasks, ptasks;
    size_t bvec_words = 0, n_lad_out = 0, cstate_words = 0, n_pbest1 = 0;
    const bool two_d = !getenv("NR_JOINT_NO_2D");
    int lad_max_t = std::max(1, (int)n_right);
    const bool ladder_on = !getenv("NR_JOINT_RECTANGLES") && n_right >= 10 && n_left >= 1;
    if (ladder_on && n_points > 0) {
        std::string rev(right, (size_t)n_right);
        std::reverse(rev.begin(), rev.end());
        const long long rev_word = pool.add(rev.data(), n_right, false);
        std::vector<std::vector<int>> of_read(n_reads);
        for (int i = 0; i < n_points; ++i) of_read[point_read[i]].push_back(i);
        std::map<std::pair<int, int>, long long> fwd_tpl;                 // (k1, k2 of the longest) -> word
        std::map<int, long long> pre_tpl, cont_tpl;                       // k1 of the longest -> left + m1*k1; k2 -> mid + m2*k2
        std::string s;
        for (int r = 0; r < n_reads && rev_word >= 0; ++r) {
            const std::vector<int>& pts = of_read[r];
            if (pts.empty() || read_len[r] < 1) continue;
            std::vector<int> K1, K2;
            for (int i : pts) { K1.push_back(point_k1[i]); K2.push_back(point_k2[i]); }
            std::sort(K1.begin(), K1.end()); K1.erase(std::unique(K1.begin(), K1.end()), K1.end());
            std::sort(K2.begin(), K2.end()); K2.erase(std::unique(K2.begin(), K2.end()), K2.end());
            if (K2.size() > (size_t)nrw::kMaxK2) continue;
            // a full grid: every (k1, k2) of K1 x K2 is among the points (duplicates allowed)
            auto idx1 = [&](int k) { return (size_t)(std::lower_bound(K1.begin(), K1.end(), k) - K1.begin()); };
            auto idx2 = [&](int k) { return (size_t)(std::lower_bound(K2.begin(), K2.end(), k) - K2.begin()); };
            std::vector<uint8_t> seen(K1.size() * K2.size(), 0);
            size_t distinct = 0;
            for (int i : pts) {
                uint8_t& c = seen[idx1(point_k1[i]) * K2.size() + idx2(point_k2[i])];
                distinct += c == 0;
                c = 1;
            }
            if (distinct != seen.size()) continue;                                   // not a full grid
            const int k2_step = K2.size() > 1 ? K2[1] - K2[0] : 1;
            bool arithmetic = true;
            for (size_t j = 1; j < K2.size(); ++j) arithmetic = arithmetic && K2[j] - K2[j - 1] == k2_step;
            if (!arithmetic) continue;
            const long long t_max = (long long)n_left + (long long)m1 * K1.back() + n_mid + (long long)m2 * K2.back();
            if (t_max + n_right > kMaxTlen || t_max + 10 - win_a > kMaxWindow ||
                (long long)sc->match * std::min<long long>(read_len[r], t_max + n_right) > kMaxScore)
                continue;                                                            // the rectangle path decides (and skips) these
            // 2-D: K1 arithmetic as well, a first junction with at least one column of its own, the saved columns within budget
            const int k1_step = K1.size() > 1 ? K1[1] - K1[0] : 1;
            bool share_k1 = two_d && K1.size() >= 2 && K1.size() <= (size_t)nrw::kMaxK2 && n_mid + m2 * K2[0] >= 1 &&
                            cstate_words + 6 * K1.size() * (size_t)read_len[r] < ((size_t)1 << 29);
            for (size_t j = 1; j < K1.size(); ++j) share_k1 = share_k1 && K1[j] - K1[j - 1] == k1_step;
            long long pre_word = -1, cont_word = -1;
            if (share_k1) {
                auto ip = pre_tpl.find(K1.back());
                if (ip == pre_tpl.end()) {
                    s.assign(left, (size_t)n_left);
                    for (int u = 0; u < K1.back(); ++u) s.append(motif1, (size_t)m1);
                    ip = pre_tpl.emplace(K1.back(), pool.add(s.data(), (int)s.size(), false)).first;
                }
                auto ic = cont_tpl.find(K2.back());
                if (ic == cont_tpl.end()) {
                    s.assign(mid ? mid : "", (size_t)n_mid);
                    for (int u = 0; u < K2.back(); ++u) s.append(motif2, (size_t)m2);
                    ic = cont_tpl.emplace(K2.back(), pool.add(s.data(), (int)s.size(), false)).first;
                }
                pre_word = ip->second; cont_word = ic->second;
                share_k1 = pre_word >= 0 && cont_word >= 0;
            }
            bool ok = true;
            std::vector<long long> words(K1.size());
            for (size_t a = 0; a < K1.size() && ok && !share_k1; ++a) {
                auto key = std::make_pair(K1[a], K2.back());
                auto it = fwd_tpl.find(key);
                if (it == fwd_tpl.end()) {
                    s.assign(left, (size_t)n_left);
                    for (int u = 0; u < K1[a]; ++u) s.append(motif1, (size_t)m1);
                    s.append(mid ? mid : "", (size_t)n_mid);
                    for (int u = 0; u < K2.back(); ++u) s.append(motif2, (size_t)m2);
                    it = fwd_tpl.emplace(key, pool.add(s.data(), (int)s.size(), false)).first;
                }
                words[a] = it->second;
                ok = words[a] >= 0;
            }
            if (!ok) continue;
            const int b0 = (int)btasks.size();
            for (int sd = 0; sd < 2; ++sd) {
                nrw::LadBwdTask bt = {};
                bt.q_word = (uint32_t)read_word[r]; bt.q_len = read_len[r];
                bt.rev_word = (uint32_t)rev_word; bt.n_right = n_right;
                bt.reverse = sd; bt.set_bvec_off((long long)bvec_words);
                bvec_words += 3 * (size_t)read_len[r];
                btasks.push_back(bt);
            }
            std::vector<int> slot(K1.size(), 0);                                     // k1 index -> first record of strand '+'
            int pre_pbest[2] = {0, 0};
            long long pre_cstate[2] = {0, 0};
            if (share_k1)
                for (int sd = 0; sd < 2; ++sd) {
                    nrw::LadFwdTask pt = {};
                    pt.q_word = (uint32_t)read_word[r]; pt.q_len = read_len[r];
                    pt.t_word = (uint32_t)pre_word;
                    pt.n_pre = n_left; pt.m2 = m1; pt.k2_first = K1[0]; pt.k2_step = k1_step; pt.k2_count = (int)K1.size();
                    pt.win_a = win_a; pt.reverse = sd; pt.bwd = b0 + sd; pt.mode = nrw::kPrefix;
                    pt.out_off = pre_pbest[sd] = (int)n_pbest1;
                    pt.cstate = pre_cstate[sd] = (long long)cstate_words;
                    n_pbest1 += K1.size();
                    cstate_words += 3 * K1.size() * (size_t)read_len[r];
                    lad_max_t = std::max(lad_max_t, n_left + m1 * K1.back());
                    ptasks.push_back(pt);
                }
            for (size_t a = 0; a < K1.size(); ++a)
                for (int sd = 0; sd < 2; ++sd) {
                    nrw::LadFwdTask ft = {};
                    ft.q_word = (uint32_t)read_word[r]; ft.q_len = read_len[r];
                    if (share_k1) {
                        ft.t_word = (uint32_t)cont_word;
                        ft.n_pre = n_mid;
                        ft.mode = nrw::kCont;
                        ft.pbest1 = pre_pbest[sd] + (int)a;
                        ft.cstate = pre_cstate[sd] + (long long)(3 * a) * read_len[r];
                    } else {
                        ft.t_word = (uint32_t)words[a];
                        ft.n_pre = n_left + m1 * K1[a] + n_mid;
                        ft.mode = nrw::kWhole;
                    }
                    ft.m2 = m2; ft.k2_first = K2[0]; ft.k2_step = k2_step; ft.k2_count = (int)K2.size();
                    ft.win_a = win_a; ft.reverse = sd; ft.bwd = b0 + sd; ft.out_off = (int)n_lad_out;
                    if (sd == 0) slot[a] = (int)n_lad_out;
                    n_lad_out += K2.size();
                    lad_max_t = std::max(lad_max_t, ft.n_pre + m2 * K2.back());
                    ftasks.push_back(ft);
                }
            for (int i : pts) {
                by_ladder[i] = 1;
                point_slot[i] = slot[idx1(point_k1[i])] + (int)idx2(point_k2[i]);
                point_slot_rev[i] = point_slot[i] + (int)K2.size();
            }
        }
    }
    mark("tasks of the shared sweeps");
    if (!ftasks.empty()) {
        // out_off, pbest1 and bwd are 32-bit task fields (bvec_off and cstate are 64-bit)
        if (n_lad_out > (size_t)INT_MAX || n_pbest1 > (size_t)INT_MAX || btasks.size() > (size_t)INT_MAX ||
            ftasks.size() > (size_t)INT_MAX)
            return nri::fail_msg(NR_ERR_ARG, "nr_joint_grid: more than 2^31 records of the shared sweeps in one call");
        if ((rc = check_pool(pool, "nr_joint_grid: more than 2^32 words of packed sequence in one call"))) return rc;
        std::vector<int2> res;
        if ((rc = run_ladder_tasks(sc, btasks, ptasks, ftasks, pool, bvec_words, cstate_words, n_pbest1, n_lad_out, lad_max_t, res, launches)))
            return rc;
        for (int i = 0; i < n_points; ++i) {
            if (!by_ladder[i]) continue;
            const int2 f = res[point_slot[i]], v = res[point_slot_rev[i]];
            const bool rev = v.x > f.x || (v.x == f.x && v.y > f.y);
            out[i].score = rev ? v.x : f.x;
            out[i].window_score = rev ? v.y : f.y;
            if (strand) strand[i] = rev ? 1 : 0;
        }
    }

    mark("shared sweeps + results");
    // ---- one template per distinct remaining grid point: left + motif1 * k1 + mid + motif2 * k2 + right (nanoRepeat_joint.py:351-374)
    std::map<std::pair<int, int>, std::pair<long long, int>> tpl;      // (k1, k2) -> (word, length)
    std::vector<nrw::WinTask> tasks;
    std::vector<int> task_point;
    std::vector<uint8_t> no_tpl;                                      // per grid point: its template holds a base other than ACGT
    std::string s;
    for (int i = 0; i < n_points; ++i) {
        if (by_ladder[i]) continue;
        const int r = point_read[i], k1 = point_k1[i], k2 = point_k2[i];
        auto key = std::make_pair(k1, k2);
        auto it = tpl.find(key);
        if (it == tpl.end()) {
            s.assign(left ? left : "", (size_t)n_left);
            for (int u = 0; u < k1; ++u) s.append(motif1, (size_t)m1);
            s.append(mid ? mid : "", (size_t)n_mid);
            for (int u = 0; u < k2; ++u) s.append(motif2, (size_t)m2);
            s.append(right ? right : "", (size_t)n_right);
            it = tpl.emplace(key, std::make_pair(pool.add(s.data(), (int)s.size(), false), (int)s.size())).first;
        }
        const long long tw = it->second.first;
        const int tl = it->second.second;
        nrw::WinTask t = {};
        t.q_word = (uint32_t)read_word[r]; t.q_len = read_len[r];
        t.t_word = tw < 0 ? 0u : (uint32_t)tw; t.t_len = tw < 0 ? 0 : tl;
        t.win_a = win_a;
        t.win_b = std::min(n_left + m1 * k1 + n_mid + m2 * k2 + 10, tl);
        t.reverse = 0; tasks.push_back(t);
        t.reverse = 1; tasks.push_back(t);
        task_point.push_back(i);
        no_tpl.push_back(tw < 0);
    }
    std::vector<nr_window_t> res(tasks.size());
    std::vector<uint8_t> skipped(tasks.size(), 0);
    for (size_t j = 0; j < tasks.size(); ++j) skipped[j] = no_tpl[j / 2];
    if ((rc = run_window_tasks(sc, tasks, pool, res.data(), skipped, launches))) return rc;
    st.kernel_launches = launches;
    for (size_t j = 0; j < task_point.size(); ++j) {
        const int i = task_point[j];
        st.n_skipped += skipped[2 * j] | skipped[2 * j + 1];                       // once per grid point
        const nr_window_t f = res[2 * j], v = res[2 * j + 1];
        // the better strand by (score, window score); '+' on a full tie
        const bool rev = v.score > f.score || (v.score == f.score && v.window_score > f.window_score);
        out[i] = rev ? v : f;
        if (strand) strand[i] = rev ? 1 : 0;
    }
    nri::set_last_stats(st);
    return NR_OK;
}
