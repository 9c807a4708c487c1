// nr_joint.cu -- host side of the joint path (nanoRepeat-joint): alignment score and window score of every (read,
// template) task in one DP (nr_window_kernel.cuh, nr_window_ladder.cuh; launched by nr_launch_window.cu).
// C ABI: nr_window_tasks, nr_joint_grid.
#include "nr_internal.h"
#include "nr_launch_window.h"

#include <algorithm>
#include <climits>
#include <map>
#include <string>
#include <tuple>
#include <vector>

namespace {

// The joint path's limits (include/nanorepeat_b200.h): the DP word holds score * 65536 + payload, so the score must stay
// within 15 bits (nri::kMaxScore) and the window within 8 000 bases (payload <= +16 000); the per-warp scratch row holds
// one template.
constexpr int kMaxWindow = 8000, kMaxTlen = 1 << 20;

// Every pool word a kernel reads through a 32-bit task field must fit it.
int check_pool(const nri::Pool& pool, const char* who) {
    if (pool.words.size() + 4 > (size_t)UINT32_MAX)
        return nri::fail(NR_ERR_ARG, "%s: more than 2^32 words of packed sequence in one call", who);
    return NR_OK;
}

nrw::WinScore window_score_words(const nr_scoring_t* sc) {
    nrw::WinScore k;
    k.match = sc->match << 16; k.mismatch = -(sc->mismatch << 16); k.ambiguous = -(sc->ambiguous << 16);
    k.open1 = -((sc->gap_open1 + sc->gap_ext1) << 16); k.ext1 = -(sc->gap_ext1 << 16);
    k.open2 = -((sc->gap_open2 + sc->gap_ext2) << 16); k.ext2 = -(sc->gap_ext2 << 16);
    return k;
}

// thread blocks of a launch over n tasks, one warp per task: at most two per SM
int warp_blocks(int n) { return std::max(1, std::min(2 * nri::sm_count(), (n + nrw::kWarps - 1) / nrw::kWarps)); }

// int4 per warp of the scratch: two rows (one per stripe parity) of the longest template
int scratch_stride(int max_t) { return 2 * ((max_t + 31) / 32 * 32); }

// tasks[i].q_word / t_word index `pool`; out[i] = (score, window score).  skipped[i] (in: 1 for a template the pool could
// not pack) is set for every task beyond the limits above; a skipped task is not scored and its record stays (0, 0).
int run_window_tasks(const nr_scoring_t* sc, std::vector<nrw::WinTask>& tasks, const nri::Pool& pool, nr_window_t* out,
                     std::vector<uint8_t>& skipped, int& launches) {
    const int n = (int)tasks.size();
    if (n == 0) return NR_OK;
    if (int rc = check_pool(pool, "joint path")) return rc;
    int max_t = 1;
    for (int i = 0; i < n; ++i) {
        nrw::WinTask& t = tasks[i];
        const long long m = (long long)sc->match * std::min(t.q_len, t.t_len);
        if (m > nri::kMaxScore || t.win_b - t.win_a > kMaxWindow || t.t_len > kMaxTlen) { t.q_len = 0; skipped[i] = 1; }
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
    const int blocks = warp_blocks(n), stride = scratch_stride(max_t);
    const size_t task_bytes = sizeof(nrw::WinTask) * n, out_bytes = sizeof(int2) * n;
    nri::Bufs bufs;
    void *d_tasks = nullptr, *d_pool = nullptr, *d_out = nullptr, *d_scratch = nullptr, *d_counter = nullptr, *h_out = nullptr;
    int rc;
    if ((rc = bufs.get(&d_tasks, task_bytes, false)) || (rc = bufs.get(&d_pool, sizeof(uint32_t) * (pool.words.size() + 4), false)) ||
        (rc = bufs.get(&d_out, out_bytes, false)) ||
        (rc = bufs.get(&d_scratch, sizeof(int4) * (size_t)blocks * nrw::kWarps * stride, false)) ||
        (rc = bufs.get(&d_counter, 256, false)) || (rc = bufs.get(&h_out, out_bytes, true)))
        return rc;
    cudaStream_t st = nri::stream();
    CUDA_TRY(cudaMemcpyAsync(d_tasks, sorted.data(), task_bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_pool, pool.words.data(), sizeof(uint32_t) * pool.words.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(d_counter, 0, 256, st));
    CUDA_TRY(nrl::launch_window(blocks, st, static_cast<const nrw::WinTask*>(d_tasks), n, static_cast<const uint32_t*>(d_pool),
                                window_score_words(sc), static_cast<int4*>(d_scratch), stride, static_cast<int*>(d_counter),
                                static_cast<int2*>(d_out)));
    ++launches;
    CUDA_TRY(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const int2* res = static_cast<const int2*>(h_out);
    for (int i = 0; i < n; ++i) { out[order[i]].score = res[i].x; out[order[i]].window_score = res[i].y; }
    return NR_OK;
}

// s += prefix + motif * k
void add_repeat(std::string& s, const char* prefix, int n_prefix, const char* motif, int m, int k) {
    if (n_prefix > 0) s.append(prefix, (size_t)n_prefix);
    for (int u = 0; u < k; ++u) s.append(motif, (size_t)m);
}

// The common difference of sorted distinct values (1 for a single value), 0 if they are not an arithmetic progression
int common_step(const std::vector<int>& K) {
    const int step = K.size() > 1 ? K[1] - K[0] : 1;
    for (size_t j = 1; j < K.size(); ++j)
        if (K[j] - K[j - 1] != step) return 0;
    return step;
}

// One nr_joint_grid call: the locus  left + motif1*k1 + mid + motif2*k2 + right  (nanoRepeat_joint.py:351-374), its reads
// and grid points, and what the stages below build from them.  Every grid point gets two records in `rec`, one per
// strand: from the shared sweeps (nr_window_ladder.cuh) for the reads whose points form a full grid, from one rectangle
// per template (nr_window_kernel.cuh) for the rest.
struct JointGrid {
    const nr_scoring_t* sc;
    const char *left, *mid, *right, *motif1, *motif2;
    int n_left, n_mid, n_right, m1, m2;
    int n_reads; const char* const* reads; const int32_t* read_len;
    int n_points; const int32_t *point_read, *point_k1, *point_k2;

    nri::Pool pool;
    std::vector<long long> read_word;
    std::vector<nr_window_t> rec;
    std::vector<long long> rec_plus, rec_minus;      // per grid point: its records of strands '+' and '-' (-1: none yet)
    // the shared sweeps: backward, prefix and forward tasks, and the sizes of their device arrays
    std::vector<nrw::LadBwdTask> btasks;
    std::vector<nrw::LadFwdTask> ftasks, ptasks;
    size_t bvec_words = 0, n_lad_out = 0, cstate_words = 0, n_pbest1 = 0;
    int lad_max_t = 1;
    // templates packed so far: (parts, k1, k2) -> (word, length); word -1: a base other than ACGT
    enum { kFirst = 1, kSecond = 2, kRight = 4 };    // parts: left + motif1*k1, mid + motif2*k2, right
    std::map<std::tuple<int, int, int>, std::pair<long long, int>> tpl_of;
    std::string s;

    int win_a = std::max(n_left - 10, 0);        // window start of every grid point (nanoRepeat_joint.py:448-451)

    std::pair<long long, int> tpl(int parts, int k1, int k2) {
        const auto key = std::make_tuple(parts, k1, k2);
        auto it = tpl_of.find(key);
        if (it == tpl_of.end()) {
            s.clear();
            if (parts & kFirst) add_repeat(s, left, n_left, motif1, m1, k1);
            if (parts & kSecond) add_repeat(s, mid, n_mid, motif2, m2, k2);
            if ((parts & kRight) && n_right > 0) s.append(right, (size_t)n_right);
            it = tpl_of.emplace(key, std::make_pair(pool.add(s.data(), (int)s.size(), false), (int)s.size())).first;
        }
        return it->second;
    }

    // ---- stage 1: the reads into the pool
    int pack_reads() {
        size_t words = 0;
        for (int r = 0; r < n_reads; ++r) words += (size_t)(std::max(read_len[r], 0) + 15) / 16 + 2;
        pool.words.reserve(words + 4096);
        read_word.resize(n_reads);
        for (int r = 0; r < n_reads; ++r) {
            if (read_len[r] < 0) return nri::fail(NR_ERR_ARG, "nr_joint_grid: negative read length");
            read_word[r] = pool.add(reads[r], read_len[r], true);
        }
        rec_plus.assign(n_points, -1);
        rec_minus.assign(n_points, -1);
        return NR_OK;
    }

    // ---- stage 2: the shared sweeps of every read whose points are a full K1 x K2 grid with K2 an arithmetic progression
    // (what joint.py's round-2 and round-3 grids are); everything else is scored template by template (stage 3).
    void plan_sweeps() {
        if (getenv("NR_JOINT_RECTANGLES") || n_right < 10 || n_left < 1 || n_points == 0) return;
        lad_max_t = std::max(1, n_right);
        std::string rev(right, (size_t)n_right);
        std::reverse(rev.begin(), rev.end());
        const long long rev_word = pool.add(rev.data(), n_right, false);
        if (rev_word < 0) return;
        const bool two_d = !getenv("NR_JOINT_NO_2D");
        std::vector<std::vector<int>> of_read(n_reads);
        for (int i = 0; i < n_points; ++i) of_read[point_read[i]].push_back(i);
        for (int r = 0; r < n_reads; ++r)
            if (!of_read[r].empty() && read_len[r] >= 1) plan_read(r, of_read[r], rev_word, two_d);
    }

    void plan_read(int r, const std::vector<int>& pts, long long rev_word, bool two_d) {
        std::vector<int> K1, K2;
        for (int i : pts) { K1.push_back(point_k1[i]); K2.push_back(point_k2[i]); }
        std::sort(K1.begin(), K1.end()); K1.erase(std::unique(K1.begin(), K1.end()), K1.end());
        std::sort(K2.begin(), K2.end()); K2.erase(std::unique(K2.begin(), K2.end()), K2.end());
        if (K2.size() > (size_t)nrw::kMaxK2) return;
        // a full grid: every (k1, k2) of K1 x K2 is among the points (duplicates allowed)
        auto idx1 = [&](int k) { return (size_t)(std::lower_bound(K1.begin(), K1.end(), k) - K1.begin()); };
        auto idx2 = [&](int k) { return (size_t)(std::lower_bound(K2.begin(), K2.end(), k) - K2.begin()); };
        std::vector<uint8_t> seen(K1.size() * K2.size(), 0);
        size_t n_seen = 0;
        for (int i : pts) {
            uint8_t& c = seen[idx1(point_k1[i]) * K2.size() + idx2(point_k2[i])];
            n_seen += c == 0;
            c = 1;
        }
        if (n_seen != seen.size()) return;                                       // not a full grid
        const int k2_step = common_step(K2);
        if (k2_step == 0) return;
        const long long t_max = (long long)n_left + (long long)m1 * K1.back() + n_mid + (long long)m2 * K2.back();
        if (t_max + n_right > kMaxTlen || t_max + 10 - win_a > kMaxWindow ||
            (long long)sc->match * std::min<long long>(read_len[r], t_max + n_right) > nri::kMaxScore)
            return;                                                               // the rectangles decide (and skip) these
        // 2-D: K1 arithmetic as well, a first junction with at least one column of its own, the saved columns within budget
        const int k1_step = common_step(K1);
        bool share_k1 = two_d && K1.size() >= 2 && K1.size() <= (size_t)nrw::kMaxK2 && k1_step != 0 && n_mid + m2 * K2[0] >= 1 &&
                        cstate_words + 6 * K1.size() * (size_t)read_len[r] < ((size_t)1 << 29);
        long long pre_word = -1, cont_word = -1;
        if (share_k1) {
            pre_word = tpl(kFirst, K1.back(), 0).first;
            cont_word = tpl(kSecond, 0, K2.back()).first;
            share_k1 = pre_word >= 0 && cont_word >= 0;
        }
        std::vector<long long> words(K1.size());
        for (size_t a = 0; a < K1.size() && !share_k1; ++a)
            if ((words[a] = tpl(kFirst | kSecond, K1[a], K2.back()).first) < 0) return;
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
            rec_plus[i] = slot[idx1(point_k1[i])] + (long long)idx2(point_k2[i]);
            rec_minus[i] = rec_plus[i] + (long long)K2.size();
        }
    }

    // ---- stage 4a: the shared sweeps (backward tasks, then prefix and forward tasks) -> rec[0, n_lad_out)
    int run_sweeps(int& launches) {
        const int nb = (int)btasks.size(), nf = (int)ftasks.size(), np = (int)ptasks.size();
        if (nf == 0) return NR_OK;
        // out_off, pbest1 and bwd are 32-bit task fields (bvec_off and cstate are 64-bit)
        if (n_lad_out > (size_t)INT_MAX || n_pbest1 > (size_t)INT_MAX || btasks.size() > (size_t)INT_MAX || ftasks.size() > (size_t)INT_MAX)
            return nri::fail(NR_ERR_ARG, "nr_joint_grid: more than 2^31 records of the shared sweeps in one call");
        if (int rc = check_pool(pool, "nr_joint_grid")) return rc;
        // long tasks first
        auto by_cost = [](const nrw::LadFwdTask& x, const nrw::LadFwdTask& y) {
            const long long cx = (long long)x.q_len * (x.n_pre + (long long)x.m2 * (x.k2_first + (long long)x.k2_step * (x.k2_count - 1)));
            const long long cy = (long long)y.q_len * (y.n_pre + (long long)y.m2 * (y.k2_first + (long long)y.k2_step * (y.k2_count - 1)));
            return cx != cy ? cx > cy : x.out_off < y.out_off;
        };
        std::sort(ftasks.begin(), ftasks.end(), by_cost);
        std::sort(ptasks.begin(), ptasks.end(), by_cost);
        const int blocks_b = warp_blocks(nb), blocks_f = warp_blocks(nf), blocks_p = warp_blocks(np);
        const int stride = scratch_stride(lad_max_t);
        const size_t scratch_bytes = sizeof(int4) * (size_t)std::max(std::max(blocks_b, blocks_f), blocks_p) * nrw::kWarps * stride;
        const size_t out_bytes = sizeof(int2) * n_lad_out;
        nri::Bufs bufs;
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
        const auto* bt = static_cast<const nrw::LadBwdTask*>(d_b);
        const auto* pool_dev = static_cast<const uint32_t*>(d_pool);
        int* counter = static_cast<int*>(d_counter);
        CUDA_TRY(cudaMemcpyAsync(d_b, btasks.data(), sizeof(nrw::LadBwdTask) * nb, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(d_f, ftasks.data(), sizeof(nrw::LadFwdTask) * nf, cudaMemcpyHostToDevice, st));
        if (np) CUDA_TRY(cudaMemcpyAsync(d_p, ptasks.data(), sizeof(nrw::LadFwdTask) * np, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(d_pool, pool.words.data(), sizeof(uint32_t) * pool.words.size(), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemsetAsync(d_counter, 0, 256, st));
        CUDA_TRY(nrl::launch_ladder_bwd(blocks_b, st, bt, nb, pool_dev, k, static_cast<int4*>(d_scratch), stride, counter,
                                        static_cast<int*>(d_bvec), static_cast<int*>(d_ronly)));
        ++launches;
        auto forward = [&](int blocks, const void* tasks, int n, int* task_counter) {
            return nrl::launch_ladder_fwd(blocks, st, static_cast<const nrw::LadFwdTask*>(tasks), n, bt, pool_dev, k,
                                          static_cast<int4*>(d_scratch), stride, task_counter, static_cast<const int*>(d_bvec),
                                          static_cast<const int*>(d_ronly), static_cast<int*>(d_cstate), static_cast<int*>(d_pbest1),
                                          static_cast<int2*>(d_out));
        };
        if (np) {       // prefix sweeps: the columns the continuation sweeps start from
            CUDA_TRY(forward(blocks_p, d_p, np, counter + 16));
            ++launches;
        }
        CUDA_TRY(forward(blocks_f, d_f, nf, counter + 32));
        ++launches;
        CUDA_TRY(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        const int2* res = static_cast<const int2*>(h_out);
        rec.resize(n_lad_out);
        for (size_t j = 0; j < n_lad_out; ++j) rec[j] = {res[j].x, res[j].y};
        return NR_OK;
    }

    // ---- stage 3: one template per distinct remaining grid point, left + motif1*k1 + mid + motif2*k2 + right, and a task
    // per strand (nanoRepeat_joint.py:351-374).  skipped: one entry per task, 1 for a template with a base other than ACGT.
    void plan_rectangles(std::vector<nrw::WinTask>& tasks, std::vector<uint8_t>& skipped) {
        for (int i = 0; i < n_points; ++i) {
            if (rec_plus[i] >= 0) continue;
            const int k1 = point_k1[i], k2 = point_k2[i];
            const auto [tw, tl] = tpl(kFirst | kSecond | kRight, k1, k2);
            nrw::WinTask t = {};
            t.q_word = (uint32_t)read_word[point_read[i]]; t.q_len = read_len[point_read[i]];
            t.t_word = tw < 0 ? 0u : (uint32_t)tw; t.t_len = tw < 0 ? 0 : tl;
            t.win_a = win_a;
            t.win_b = std::min(n_left + m1 * k1 + n_mid + m2 * k2 + 10, tl);
            rec_plus[i] = (long long)(n_lad_out + tasks.size());
            rec_minus[i] = rec_plus[i] + 1;
            t.reverse = 0; tasks.push_back(t);
            t.reverse = 1; tasks.push_back(t);
            skipped.push_back(tw < 0); skipped.push_back(tw < 0);
        }
    }
};

}  // namespace

extern "C" int nr_window_tasks(const nr_scoring_t* sc, int32_t n_tasks, const char* const* queries, const int32_t* qlen,
                               const char* const* targets, const int32_t* tlen, const int32_t* win_a, const int32_t* win_b,
                               const uint8_t* reverse, nr_window_t* out) {
    if (nri::check(sc)) return nri::last_code();
    if (n_tasks < 0 || (n_tasks > 0 && (!queries || !qlen || !targets || !tlen || !win_a || !win_b || !out)))
        return nri::fail(NR_ERR_ARG, "nr_window_tasks: bad arguments");
    int rc = nri::ensure_init();
    if (rc) return rc;
    nr_stats_t st = {};
    st.n_tasks = n_tasks;
    nri::set_last_stats(st);
    nri::PhaseTrace trace;
    nri::Pool pool;
    std::vector<nrw::WinTask> tasks(n_tasks);
    std::vector<uint8_t> skipped(n_tasks, 0);
    std::map<std::pair<const char*, int>, long long> seen_q, seen_t;
    for (int i = 0; i < n_tasks; ++i) {
        nrw::WinTask& t = tasks[i];
        t = {};
        out[i].score = out[i].window_score = 0;
        if (qlen[i] < 0 || tlen[i] < 0) return nri::fail(NR_ERR_ARG, "nr_window_tasks: negative length");
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
    trace.mark("window tasks: pack");
    int launches = 0;
    rc = run_window_tasks(sc, tasks, pool, out, skipped, launches);
    trace.mark("window tasks: run");
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
        return nri::fail(NR_ERR_ARG, "nr_joint_grid: bad arguments");
    int rc = nri::ensure_init();
    if (rc) return rc;
    nr_stats_t st = {};
    st.n_tasks = n_points;
    nri::set_last_stats(st);
    nri::PhaseTrace trace;
    JointGrid g{sc, left, mid, right, motif1, motif2, n_left, n_mid, n_right, m1, m2, n_reads, reads, read_len, n_points,
                point_read, point_k1, point_k2};
    if ((rc = g.pack_reads())) return rc;
    trace.mark("joint grid: pack reads");
    for (int i = 0; i < n_points; ++i) {
        if (point_read[i] < 0 || point_read[i] >= n_reads || point_k1[i] < 0 || point_k2[i] < 0)
            return nri::fail(NR_ERR_ARG, "nr_joint_grid: bad grid point");
        out[i].score = out[i].window_score = 0;
        if (strand) strand[i] = 0;
    }
    g.plan_sweeps();
    trace.mark("joint grid: plan sweeps");
    int launches = 0;
    if ((rc = g.run_sweeps(launches))) return rc;
    trace.mark("joint grid: shared sweeps");
    std::vector<nrw::WinTask> tasks;
    std::vector<uint8_t> skipped;
    g.plan_rectangles(tasks, skipped);
    g.rec.resize(g.n_lad_out + tasks.size());
    if ((rc = run_window_tasks(sc, tasks, g.pool, g.rec.data() + g.n_lad_out, skipped, launches))) return rc;
    trace.mark("joint grid: rectangles");
    st.kernel_launches = launches;
    for (size_t j = 0; j < skipped.size(); j += 2) st.n_skipped += skipped[j] | skipped[j + 1];      // once per grid point
    // ---- stage 5: per grid point the better strand by (score, window score); '+' on a full tie
    for (int i = 0; i < n_points; ++i) {
        const nr_window_t f = g.rec[g.rec_plus[i]], v = g.rec[g.rec_minus[i]];
        const bool rev = v.score > f.score || (v.score == f.score && v.window_score > f.window_score);
        out[i] = rev ? v : f;
        if (strand) strand[i] = rev ? 1 : 0;
    }
    nri::set_last_stats(st);
    return NR_OK;
}
