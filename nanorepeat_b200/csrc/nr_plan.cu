// nr_plan.cu -- the launch plan of a committed batch, on the host and without CUDA calls: which reads share a u16x2 warp,
// the stripe heights of the long reads, their CoopInfo scratch, the entries of the 32-bit launch, every buffer size and
// the blob's sections.  nr_api.cu (upload_batch) allocates and uploads what it decided.
#include "nr_batch.h"

#include <algorithm>
#include <numeric>

namespace nrh {
namespace {

// Round 2's dominance exit (nr_pair_kernels.cuh, Sweep::run; DESIGN.md section 4.9).  NR_ROUND2_EXIT=0 turns it off
// for the batches committed while it is set (A/B measurements); it changes no result either way.
bool round2_exit_enabled() {
    const char* e = getenv("NR_ROUND2_EXIT");
    return !(e && atoi(e) == 0);
}
// A core is 100 read bases of left flank + repeat + 100 of right flank (nanoRepeat_bam.py:308-316), so its repeat
// ends near column |left| + q - 100 of the template and the DP past it turns periodic within a few motif copies.  On
// config 2 (tools/round2_exit_census.py) the sweep ends at |left| + q - 83 on average; checks from |left| + q - 192 find
// the same exits as checks from |left| on (18.1 % of the region's cells), from |left| + q - 100 they find 16.5 %.
int round2_check_col(int n_left, int q_len) { return std::max(n_left + 1, n_left + q_len - 192); }
int round2_predicted_exit(int n_left, int q_len) { return n_left + std::max(q_len - 64, 32); }

// Pair up the eligible tasks of one region (ids[]: task indices, all of the same template): neighbours in read length
// share a warp, one per 16-bit half of the DP words (nr_pair_kernels.cuh).  key(i) orders the tasks.
template <class Key, class Emit>
void make_pairs(std::vector<int>& ids, Key key, Emit emit) {
    // decreasing key, then increasing id: one 64-bit word per task, (key << 32) | ~id, sorted downwards
    std::vector<uint64_t> w(ids.size());
    for (size_t i = 0; i < ids.size(); ++i) w[i] = ((uint64_t)(uint32_t)key(ids[i]) << 32) | (uint32_t)~(uint32_t)ids[i];
    std::sort(w.begin(), w.end(), std::greater<uint64_t>());
    for (size_t i = 0; i < w.size(); ++i) ids[i] = (int)~(uint32_t)w[i];
    for (size_t i = 0; i < ids.size(); i += 2) emit(ids[i], i + 1 < ids.size() ? ids[i + 1] : -1);
}

struct LongPair { int a, b, n_left; long long cost; };

// The state the stages of one plan share.  Tasks are b->ltasks (ladder) or b->tasks.
struct Planner {
    nr_batch* b;
    const int sm_count;
    const bool ladder = b->ladder;
    const bool fixed = is_map_ont(b->sc);
    const int n = ladder ? (int)b->ltasks.size() : (int)b->tasks.size();
    const int max_r = ladder ? nr::kMaxRLadder : nr::kMaxRExact;
    Launch& L = b->launch;
    // per task: its cost in executed cells, rows per lane, stripes, columns swept and rungs
    std::vector<long long> cost = std::vector<long long>(n, 0);
    std::vector<int> task_R = std::vector<int>(n, nr::kMinR), task_ns = std::vector<int>(n, 1);
    std::vector<int> task_sweep = std::vector<int>(n, 0), task_rungs = std::vector<int>(n, 0);
    // 1: runs on the paired kernels; 2: not scored -- an empty sequence, a template that is not ACGT (t_len < 0), or a
    // task beyond the packed score / coordinate range: its record stays zero, which every caller reads as "the aligner
    // printed nothing" (nanoRepeat_bam.py:421, :433); the rest of the batch is unaffected; 3: in a pair of long reads
    std::vector<char> paired = std::vector<char>(n, 0);
    std::vector<long long> pair_cost;
    std::vector<long long> deal_cost;     // round 2: the cost the pairs are dealt by, the sweep up to the predicted exit
    long long state_off = 0;
    long long rung_off = 0;               // (P, J) token pairs of the paired ladders, single-stripe pairs first
    std::vector<LongPair> long_pairs;
    long long long_pair_rows = 0;
    std::vector<int> singles, multis;
    int coop_height = 12;
    long long data_off = 0, flag_off = 0; // CoopInfo scratch (int4) and progress flags (int) laid out so far
    std::vector<int> long_pair_ns;

    int q_len(int i) const { return ladder ? b->ltasks[i].q_len : b->tasks[i].q_len; }
    int stripes(int q, int R) const { return (q + 32 * R - 1) / (32 * R); }

    // ---- task shapes: cost, R, stripes, sweep and rungs; "not scored"; algorithmic cells ----
    void task_shapes() {
        if (b->kind != KIND_ROUND3) b->n_out = b->tasks.size();
        b->stats = {};
        b->stats.n_tasks = (int64_t)b->n_out;
        for (int i = 0; i < n; ++i) {
            int q_len, t_len, t_sweep;
            if (ladder) {
                const nr::LadderTask& t = b->ltasks[i];
                const nr::LadderRegion& g = b->lregs[t.region];
                const int flank = g.n_left + g.n_right;
                q_len = t.q_len;
                t_len = flank + g.m * t.kmax;                 // longest rung = columns swept (|R| backward, rest forward)
                t_sweep = std::max(g.n_left + g.m * t.kmax, g.n_right);
                const int rungs = t.kmax - t.kmin + 1;
                task_rungs[i] = rungs;
                b->stats.algorithmic_cells +=
                    (long long)q_len * ((long long)rungs * flank + (long long)g.m * (t.kmin + t.kmax) * rungs / 2);
            } else {
                const nr::Task& t = b->tasks[i];
                q_len = t.q_len;
                t_len = t_sweep = t.t_len;
                if (t_len > 0) b->stats.algorithmic_cells += (long long)q_len * t_len;
            }
            if (q_len <= 0 || t_len <= 0) {
                paired[i] = 2;
                if (t_len < 0) ++b->n_skipped;
                continue;
            }
            long long m = (long long)b->sc.match * std::min(q_len, t_len);
            if (m > kMaxScore || t_len > kMaxTlen) {        // (its cells stay in the count of what was asked for)
                paired[i] = 2;
                ++b->n_skipped;
                continue;
            }
            nr::stripe_shape(q_len, max_r, task_R[i], task_ns[i]);
            task_sweep[i] = t_sweep;
            cost[i] = (long long)task_ns[i] * 32 * task_R[i] * t_len;
        }
    }

    // ---- single-stripe pairs of round 2: two reads of one region per warp ----
    void pairs_round2() {
        const bool exits = round2_exit_enabled();
        for (const RegionInfo& g : b->regions) {
            std::vector<int> ids;
            for (int r = g.first_read; r < g.first_read + g.n_reads; ++r) {
                const nr::Task& t = b->tasks[r];
                if (!paired[r] && t.q_len >= 1 && t.q_len <= 32 * nr::pr::kMaxRPair2 && t.t_len >= 1) ids.push_back(r);
            }
            make_pairs(ids, [&](int i) { return b->tasks[i].q_len; }, [&](int x, int y) {
                const int R = nr::pr::pair_rows(b->tasks[x].q_len);      // x is the longer read
                nr::pr::Pair2 p = {x, y, g.n_left, -1, -1, 0, {0, 0}};
                const int t_len = b->tasks[x].t_len;
                int cols = t_len;
                if (exits) {
                    p.check_col = round2_check_col(g.n_left, b->tasks[x].q_len);
                    p.period = 16 / std::gcd(16, g.motif_len) * g.motif_len;
                    cols = std::min(t_len, round2_predicted_exit(g.n_left, b->tasks[x].q_len));
                    b->round2_exit = true;
                }
                if (g.n_left >= 2 && state_off + nr::pr::state_words(R) < 0x7fffffffLL) {
                    p.state_off = (int32_t)state_off;                    // round 3 resumes from here (nr_batch_begin_round3_from)
                    state_off += nr::pr::state_words(R);
                }
                b->pairs2.push_back(p);
                paired[x] = 1;
                if (y >= 0) paired[y] = 1;
                L.pair_R = std::max(L.pair_R, R);
                pair_cost.push_back((long long)32 * R * t_len);
                deal_cost.push_back((long long)32 * R * cols);
                b->paired_useful += (long long)(b->tasks[x].q_len + (y >= 0 ? b->tasks[y].q_len : 0)) * t_len;
            });
        }
    }

    // ---- single-stripe pairs of round 3: the pairs of the round-2 batch whose reads it reuses, then region by region ----
    int pairs_round3() {
        if (b->qsrc && !b->qsrc->pairs2.empty() && (int)b->lt_src.size() == n) {
            // the reads were paired in round 2: same pairs, same halves, same rows per lane, so that the forward sweep
            // can take over the DP state round 2 kept after column |left| - 2 instead of sweeping the left anchor again
            const nr_batch* src = b->qsrc;
            std::vector<int> src2lt(src->tasks.size(), -1);
            for (int i = 0; i < n; ++i)
                if (b->lt_src[i] >= 0) src2lt[b->lt_src[i]] = i;
            for (int pi = 0; pi < src->n_pairs2_single; ++pi) {
                const nr::pr::Pair2& p2 = src->pairs2[pi];
                int la = src2lt[p2.a], lb = p2.b >= 0 ? src2lt[p2.b] : -1;
                if (la >= 0 && paired[la]) la = -1;        // (not scored: beyond the packed range)
                if (lb >= 0 && paired[lb]) lb = -1;
                if (la < 0 && lb < 0) continue;
                const nr::LadderRegion& g = b->lregs[b->ltasks[la >= 0 ? la : lb].region];
                if (g.n_left <= 0 || g.n_right <= 0) continue;
                const int q = std::max(src->tasks[p2.a].q_len, p2.b >= 0 ? src->tasks[p2.b].q_len : 0);
                const int R = nr::pr::pair_rows(q);
                int kmin = INT32_MAX, kmax = -1;
                for (int t : {la, lb})
                    if (t >= 0) { kmin = std::min(kmin, b->ltasks[t].kmin); kmax = std::max(kmax, b->ltasks[t].kmax); }
                nr::pr::Pair3 p = {la, lb, (int32_t)rung_off, -1, R, {0, 0, 0}};
                if (p2.state_off >= 0 && src->d_state && g.n_left >= 2 && g.n_left == p2.mark_col) p.state_off = p2.state_off;
                rung_off += kmax - kmin + 1;
                b->pairs3.push_back(p);
                if (la >= 0) paired[la] = 1;
                if (lb >= 0) paired[lb] = 1;
                L.pair_R = std::max(L.pair_R, R);
                const long long cols = (long long)g.n_right + g.n_left + (long long)g.m * kmax - (p.state_off >= 0 ? g.n_left - 1 : 0);
                pair_cost.push_back((long long)32 * R * cols);
                b->paired_useful += (long long)((la >= 0 ? b->ltasks[la].q_len : 0) + (lb >= 0 ? b->ltasks[lb].q_len : 0)) * cols;
            }
        }
        for (int i0 = 0; i0 < n;) {
            int i1 = i0;
            while (i1 < n && b->ltasks[i1].region == b->ltasks[i0].region) ++i1;
            const nr::LadderRegion& g = b->lregs[b->ltasks[i0].region];
            std::vector<int> ids;
            if (g.n_left > 0 && g.n_right > 0)
                for (int i = i0; i < i1; ++i)
                    if (!paired[i] && b->ltasks[i].q_len >= 1 && b->ltasks[i].q_len <= 32 * nr::pr::kMaxRPair3) ids.push_back(i);
            make_pairs(ids, [&](int i) { return ((long long)b->ltasks[i].q_len << 20) + b->ltasks[i].kmax; }, [&](int x, int y) {
                const nr::LadderTask& tx = b->ltasks[x];
                int kmin = tx.kmin, kmax = tx.kmax;
                if (y >= 0) { kmin = std::min(kmin, b->ltasks[y].kmin); kmax = std::max(kmax, b->ltasks[y].kmax); }
                nr::pr::Pair3 p = {x, y, (int32_t)rung_off, -1, 0, {0, 0, 0}};
                rung_off += kmax - kmin + 1;
                b->pairs3.push_back(p);
                paired[x] = 1;
                if (y >= 0) paired[y] = 1;
                const int R = nr::pr::pair_rows(tx.q_len);
                L.pair_R = std::max(L.pair_R, R);
                pair_cost.push_back((long long)32 * R * (g.n_right + g.n_left + (long long)g.m * kmax));
                b->paired_useful += (long long)(tx.q_len + (y >= 0 ? b->ltasks[y].q_len : 0)) * (g.n_right + g.n_left + (long long)g.m * kmax);
            });
            i0 = i1;
        }
        if (rung_off > 0x7fffffffLL) return fail(NR_ERR_TOO_LARGE, "more than 2^31 rungs in one batch");
        L.redo_R = L.pair_R;
        return NR_OK;
    }

    // ---- pairs in decreasing (deal) cost: the tail of the persistent launch is made of the cheap ones ----
    void order_pairs() {
        L.n_pairs = (int)pair_cost.size();
        if (!L.n_pairs) return;
        std::vector<int> po(L.n_pairs);
        {
            std::vector<uint64_t> w(L.n_pairs);      // (cost << 24) | ~index: pair costs stay below 2^40, pairs below 2^24
            const std::vector<long long>& dc = deal_cost.empty() ? pair_cost : deal_cost;
            for (int i = 0; i < L.n_pairs; ++i) w[i] = ((uint64_t)dc[i] << 24) | (uint32_t)(0xffffff - i);
            std::sort(w.begin(), w.end(), std::greater<uint64_t>());
            for (int i = 0; i < L.n_pairs; ++i) po[i] = 0xffffff - (int)(w[i] & 0xffffff);
        }
        if (!b->pairs2.empty()) { std::vector<nr::pr::Pair2> t(L.n_pairs); for (int i = 0; i < L.n_pairs; ++i) t[i] = b->pairs2[po[i]]; b->pairs2.swap(t); }
        else { std::vector<nr::pr::Pair3> t(L.n_pairs); for (int i = 0; i < L.n_pairs; ++i) t[i] = b->pairs3[po[i]]; b->pairs3.swap(t); }
        for (long long c : pair_cost) b->paired_cells += 2 * c;             // both halves of every word
        b->stats.executed_cells += b->paired_cells;
        L.pair_blocks = std::max(1, std::min(sm_count, L.n_pairs));
    }

    // ---- pairs of LONG reads: two reads of a region that are longer than one paired stripe share the u16x2 words stripe
    // by stripe; their stripes are cooperative entries like the 32-bit ones.  A read pairs with the next shorter one of
    // its region (ids: the region's candidates) if that one is at least half as long (the pair sweeps the longer read's
    // rows; in round 3 the union of the two ladders).
    void pair_long_reads(std::vector<int>& ids, int n_left) {
        std::sort(ids.begin(), ids.end(), [&](int x, int y) { return q_len(x) != q_len(y) ? q_len(x) > q_len(y) : x < y; });
        for (size_t i = 0; i + 1 < ids.size();) {
            const int x = ids[i], y = ids[i + 1];
            if (2 * q_len(y) >= q_len(x)) {
                long_pairs.push_back({x, y, n_left, 0});
                paired[x] = paired[y] = 3;
                long_pair_rows += q_len(x);
                i += 2;
            } else {
                ++i;
            }
        }
    }

    void select_long_pairs() {
        std::vector<int> ids;
        if (ladder) {
            for (int i0 = 0; i0 < n;) {
                int i1 = i0;
                while (i1 < n && b->ltasks[i1].region == b->ltasks[i0].region) ++i1;
                const nr::LadderRegion& g = b->lregs[b->ltasks[i0].region];
                ids.clear();
                if (g.n_left > 0 && g.n_right > 0)
                    for (int i = i0; i < i1; ++i)
                        if (!paired[i] && b->ltasks[i].q_len > 32 * nr::pr::kMaxRPair3) ids.push_back(i);
                pair_long_reads(ids, g.n_left);
                i0 = i1;
            }
        } else {
            for (const RegionInfo& g : b->regions) {
                ids.clear();
                for (int r = g.first_read; r < g.first_read + g.n_reads; ++r)
                    if (!paired[r] && b->tasks[r].q_len > 32 * nr::pr::kMaxRPair2 && b->tasks[r].t_len >= 1) ids.push_back(r);
                pair_long_reads(ids, g.n_left);
            }
        }
    }

    // task i cut into stripes of R rows per lane (its cost scales with the rows it now sweeps)
    void restripe(int i, int R) {
        const int ns = stripes(q_len(i), R);
        cost[i] = cost[i] / ((long long)task_ns[i] * task_R[i]) * ((long long)ns * R);
        task_ns[i] = ns;
        task_R[i] = R;
    }

    // ---- the rest: one persistent launch of the 32-bit kernels.  Long reads are cut into stripes that run on different
    // warps at the same time (nr_kernels.cuh, CoopInfo).  One stripe height for the long tasks and the long pairs ----
    int stripe_heights() {
        long long multi_rows = 0;
        for (int i = 0; i < n; ++i) {
            if (paired[i]) continue;
            (task_ns[i] > 1 ? multis : singles).push_back(i);
            if (task_ns[i] > 1) multi_rows += q_len(i);
        }
        if (!multis.empty() || !long_pairs.empty()) {
            // stripe height of the long tasks: the shortest that does not cut them into more stripes than there are warps
            // to run them side by side (a stripe is one warp's work; the ladder's two sweeps overlap)
            const long long warps = (long long)nr::kWarpsPerBlock * sm_count;
            int cap = max_r;
            const char* force = getenv("NR_COOP_ROWS");       // tuning / debugging: fixed stripe height of the long tasks
            if (force && atoi(force) >= nr::kMinR && atoi(force) <= max_r) cap = std::min(nr::coop_height_at_least(atoi(force)), max_r);
            else for (int r : {4, 6, 8}) {
                if (r >= max_r) break;
                const long long st = ((multi_rows + long_pair_rows) / (32 * r) + (long long)multis.size() + (long long)long_pairs.size()) * (ladder ? 2 : 1);
                if (st <= warps) { cap = r; break; }
            }
            // ONE stripe height for all long tasks of the batch.  Every height is its own unrolled code; long reads running
            // at six different heights at once miss the instruction cache on most fetches (config 5: 4.7 stall cycles per
            // issued instruction, round 3 in 183 ms with three heights in flight against 57 ms with one).  The last stripe
            // of a task is padded up to the common height.
            coop_height = std::min(cap, 12);
            for (int i : multis) {
                int R = coop_height;
                if (stripes(q_len(i), R) > nr::kCodeFwd - 2)        // too long for that many stripes: its own, taller ones
                    R = nr::coop_height_at_least(nr::coop_rows(q_len(i), nr::kCodeFwd - 2));
                if (R > max_r)
                    return fail(NR_ERR_TOO_LARGE, "task %d: a query of %d bases needs more than %d stripes", i, q_len(i), nr::kCodeFwd - 2);
                restripe(i, R);
            }
        }
        // long pairs at the common height; one that would need more than 62 stripes goes back to the 32-bit kernels
        std::vector<LongPair> keep;
        for (LongPair& lp : long_pairs) {
            const int ns = stripes(q_len(lp.a), coop_height);
            if (ns > nr::kCodeFwd - 2 || b->pairs2.size() + b->pairs3.size() + keep.size() >= (1u << 22)) {
                for (int t : {lp.a, lp.b}) {
                    paired[t] = 0;
                    multis.push_back(t);
                    restripe(t, std::max(nr::coop_height_at_least(nr::coop_rows(q_len(t), nr::kCodeFwd - 2)), coop_height));
                }
                continue;
            }
            long long cols;
            if (ladder) {
                const nr::LadderRegion& g = b->lregs[b->ltasks[lp.a].region];
                cols = (long long)g.n_right + g.n_left + (long long)g.m * std::max(b->ltasks[lp.a].kmax, b->ltasks[lp.b].kmax);
            } else {
                cols = b->tasks[lp.a].t_len;
            }
            lp.cost = (long long)ns * 32 * coop_height * cols;
            keep.push_back(lp);
        }
        long_pairs.swap(keep);
        std::sort(long_pairs.begin(), long_pairs.end(), [](const LongPair& x, const LongPair& y) { return x.cost != y.cost ? x.cost > y.cost : x.a < y.a; });
        return NR_OK;
    }

    // Appends a CoopInfo whose scratch takes `words` int4: its data and flags follow those of the previous one.
    int add_coop(nr::CoopInfo ci, long long words) {
        ci.data_off = data_off;
        ci.flag_off = (int)flag_off;
        data_off += words;
        flag_off += nr::kCoopFlagInts(ci.n_stripes);
        if (flag_off > 0x7fffffffLL) return fail(NR_ERR_TOO_LARGE, "too many long tasks in one batch");
        b->coop.push_back(ci);
        return NR_OK;
    }

    // ---- CoopInfo of the multi-stripe tasks, then of the long pairs (those are pairs too: after the single-stripe ones) ----
    int coop_layout() {
        int rc;
        if (!ladder) b->coop_idx.assign(n, -1);
        for (int i : multis) {
            nr::CoopInfo ci = {};
            ci.n_stripes = task_ns[i];
            ci.rows = task_R[i];
            ci.bnd_stride = (task_sweep[i] + 63) / 32 * 32;
            if (ladder) {
                ci.b_stride = task_ns[i] * 32 * task_R[i];
                ci.tok_stride = (task_rungs[i] + 1) / 2 * 2;
            }
            if ((rc = add_coop(ci, (ladder ? 4LL : 2LL) * ci.bnd_stride + ci.b_stride + 2LL * ci.tok_stride))) return rc;
            if (ladder) b->ltasks[i].pad = (int32_t)b->coop.size() - 1;
            else b->coop_idx[i] = (int32_t)b->coop.size() - 1;
        }
        for (const LongPair& lp : long_pairs) {
            const int ta = lp.a, tb = lp.b, coop = (int)b->coop.size();
            nr::CoopInfo ci = {};
            ci.n_stripes = stripes(q_len(ta), coop_height);
            ci.rows = coop_height;
            if (ladder) {
                const nr::LadderTask& a = b->ltasks[ta];
                const nr::LadderRegion& g = b->lregs[a.region];
                const int kmin = std::min(a.kmin, b->ltasks[tb].kmin), kmax = std::max(a.kmax, b->ltasks[tb].kmax), rungs = kmax - kmin + 1;
                ci.bnd_stride = (std::max(g.n_left + g.m * kmax, g.n_right) + 63) / 32 * 32;
                ci.b_stride = ci.n_stripes * 32 * coop_height;          // words per plane of the backward stripes' junction state
                ci.tok_stride = (rungs + 1) / 2 * 2;
                if ((rc = add_coop(ci, 4LL * ci.bnd_stride + (3LL * ci.b_stride + 3) / 4 + 2LL * ci.tok_stride))) return rc;
                b->pairs3.push_back({ta, tb, (int32_t)rung_off, -1, coop_height, {coop, 0, 0}});
                rung_off += rungs;
                b->paired_useful += (long long)(q_len(ta) + q_len(tb)) * (lp.cost / ((long long)ci.n_stripes * 32 * coop_height));
            } else {
                ci.bnd_stride = (b->tasks[ta].t_len + 63) / 32 * 32;
                if ((rc = add_coop(ci, 2LL * ci.bnd_stride))) return rc;
                b->pairs2.push_back({ta, tb, lp.n_left, coop});      // state_off = the pair's CoopInfo
                b->paired_useful += (long long)(q_len(ta) + q_len(tb)) * b->tasks[ta].t_len;
            }
            long_pair_ns.push_back(ci.n_stripes);
            L.pair_R = std::max(L.pair_R, coop_height);
            b->paired_cells += 2 * lp.cost;
            b->stats.executed_cells += 2 * lp.cost;
        }
        b->n_long_pairs = (int)long_pairs.size();
        return NR_OK;
    }

    // ---- entries of the 32-bit launch: the long tasks' stripes, stripe-major, then the single-stripe tasks ----
    int entries() {
        int rmax = 0;
        for (int i = 0; i < n; ++i) {
            if (paired[i]) continue;
            rmax = std::max(rmax, task_R[i]);
            b->rest_cells += cost[i];
            b->rest_useful += cost[i] / ((long long)task_ns[i] * 32 * task_R[i]) * q_len(i);
        }
        b->stats.executed_cells += b->rest_cells;
        auto by_cost = [&](int x, int y) { return cost[x] != cost[y] ? cost[x] > cost[y] : x < y; };
        std::sort(singles.begin(), singles.end(), by_cost);
        std::sort(multis.begin(), multis.end(), by_cost);
        if (n > (1 << (31 - nr::kCodeBits))) return fail(NR_ERR_TOO_LARGE, "more than 2^24 tasks in one batch");
        b->order.clear();
        b->coop.clear();
        int rc;
        if ((rc = coop_layout())) return rc;
        if (rung_off > 0x7fffffffLL) return fail(NR_ERR_TOO_LARGE, "more than 2^31 rungs in one batch");
        if (!b->pairs3.empty()) b->prung_bytes = sizeof(uint2) * (size_t)std::max<long long>(rung_off, 1);
        // Stripe-major: stripe 0 of every long task, then stripe 1 of every long task, ...  A stripe waits for the one
        // above it; listed task by task, all stripes of a task would be picked up at the same moment and stripe s would
        // spin for s x (lag of ~95 columns) before its first column -- with 20 stripes over the 1000 columns of the right
        // anchor that is more waiting than work (measured on config 5: a fifth of all executed instructions were retry
        // loops).  Level by level, a stripe is picked up when the one above it is well under way or done, and the
        // parallelism comes from the tasks; with few long tasks all levels are in flight at once and the stripes pipeline
        // as before.
        const int first_long_pair = ladder ? b->n_pairs3_single : b->n_pairs2_single;
        int max_ns = 0;
        for (int i : multis) max_ns = std::max(max_ns, task_ns[i]);
        for (int ns : long_pair_ns) max_ns = std::max(max_ns, ns);
        for (int fwd = 0; fwd < (ladder ? 2 : 1); ++fwd)       // first sweep of every long task (ladder: backward), then
            for (int st = 0; st < max_ns; ++st) {               // the ladder's forward sweeps
                const int code = fwd ? nr::kCodeFwd + st : 1 + st;
                for (size_t k = 0; k < long_pair_ns.size(); ++k)    // (pairs of long reads: entries point into pairs[])
                    if (st < long_pair_ns[k]) b->order.push_back(nr::pr::kPairEntry | ((first_long_pair + (int)k) << nr::kCodeBits) | code);
                for (int i : multis)
                    if (st < task_ns[i] && (fwd || !ladder || b->lregs[b->ltasks[i].region].n_right > 0))
                        b->order.push_back((i << nr::kCodeBits) | code);
            }
        for (int i : singles) b->order.push_back(i << nr::kCodeBits);
        L.ladder = ladder;
        L.R = rmax;
        L.count = (int)b->order.size();
        // one persistent block per SM (every block resident: entries may wait for each other); a small batch still spreads
        L.blocks = std::max(1, std::min(sm_count, L.count));
        L.fixed = fixed;
        b->flags_bytes = sizeof(int) * (size_t)flag_off;
        return NR_OK;
    }

    // ---- buffer sizes and the blob: [tasks | regions | order | pairs | coop | coop_idx | pool (+4 slack words) | counters] ----
    void buffers_and_blob() {
        Section* s = b->blob;
        s[SEC_TASKS] = ladder ? Section{b->ltasks.data(), sizeof(nr::LadderTask) * n} : Section{b->tasks.data(), sizeof(nr::Task) * n};
        s[SEC_LREGS] = {b->lregs.data(), sizeof(nr::LadderRegion) * b->lregs.size()};
        s[SEC_ORDER] = {b->order.data(), sizeof(int32_t) * b->order.size()};
        s[SEC_PAIRS] = b->pairs2.empty() ? Section{b->pairs3.data(), sizeof(nr::pr::Pair3) * b->pairs3.size()}
                                         : Section{b->pairs2.data(), sizeof(nr::pr::Pair2) * b->pairs2.size()};
        s[SEC_COOP] = {b->coop.data(), sizeof(nr::CoopInfo) * b->coop.size()};
        s[SEC_COOP_IDX] = {b->coop_idx.data(), b->coop.empty() ? 0 : sizeof(int32_t) * b->coop_idx.size()};
        s[SEC_POOL] = {b->pool.words.data(), sizeof(uint32_t) * b->pool.words.size(), 16};
        size_t off = 0, h2d = 0;
        for (int k = 0; k < kBlobSections; ++k) {
            s[k].off = off;
            off += align_up(s[k].bytes + s[k].zeros, 256);
            h2d += s[k].bytes + s[k].zeros;
        }
        b->blob_bytes = off + 256;
        b->out_bytes = sizeof(int4) * std::max<size_t>(b->n_out, 1);
        b->scratch_bytes = sizeof(int4) * (size_t)data_off;
        if (b->flag) b->sel_bytes = sizeof(int4) * std::max<size_t>((size_t)b->n_reads, 1);
        if (!b->pairs3.empty()) b->redo_bytes = sizeof(int32_t) * (size_t)n * 2;   // [n] entries of the device-side redo launch | [n] long reads for the host
        b->stats.h2d_bytes = (int64_t)h2d;
        b->stats.d2h_bytes = (int64_t)sizeof(int4) * (b->flag ? (int64_t)b->n_reads : (int64_t)b->n_out);
        b->stats.n_skipped = b->n_skipped;
    }
};

}  // namespace

// Pair the eligible tasks, sort the rest (single-stripe | multi-stripe groups, each by decreasing cost), size the
// launches and the buffers.
int plan_batch(nr_batch* b, int sm_count) {
    Planner p{b, sm_count};
    PhaseTrace trace;
    int rc;
    p.task_shapes();
    trace.mark("task shapes");
    b->launch = {};
    if (b->pair && p.fixed && !p.ladder && b->kind == KIND_ROUND2) p.pairs_round2();
    else if (b->pair && p.fixed && p.ladder && b->flag && (rc = p.pairs_round3())) return rc;
    trace.mark("pairing");
    b->state_bytes = sizeof(uint32_t) * 32 * (size_t)p.state_off;
    p.order_pairs();
    trace.mark("pair order");
    b->n_pairs2_single = (int)b->pairs2.size();
    b->n_pairs3_single = (int)b->pairs3.size();
    if (b->pair && p.fixed && (p.ladder ? b->flag : b->kind == KIND_ROUND2) && !getenv("NR_NO_LONG_PAIRS")) p.select_long_pairs();
    if ((rc = p.stripe_heights()) || (rc = p.entries())) return rc;
    trace.mark("32-bit entries");
    p.buffers_and_blob();
    return NR_OK;
}

}  // namespace nrh
