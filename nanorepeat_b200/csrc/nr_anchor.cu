// nr_anchor.cu -- Step 1 of the reference's per-region pipeline for any number of regions in one call (nr_anchor_regions):
// find both anchors in every raw read and derive the core / middle positions (nanoRepeat_bam.py:165-234).
//
// Two launches, whatever the number of regions:
//   1. anchor_pair_kernel (nr_launch_anchor.cu): per read strand, both anchors on u16x2 words -> per anchor and strand
//      the exact (score, tend) of the contract (oracle/nr_oracle.c).  The words carry no start column.
//   2. the exact 32-bit kernel (a task batch of nr_api.cu) recovers qstart where the rules need it: the best hit of every
//      good anchor, scored again on the window read[a, tend) of its strand, a = max(0, tend - W),
//          W = n + max(0, floor((match * n - S - min(q, q2)) / min(e, e2))),   n = |anchor|, S = the hit's score.
//      An alignment of score S spans at most W read bases (a deletion run of length l costs at least
//      l * min(e, e2) + min(q, q2)), and tend is the smallest end reaching S on the whole strand, so every alignment of
//      the window that reaches S ends at tend: the window's record is (S, tstart - a, tend - a) with the contract's
//      tie-break.  The library checks score and end and fails the call rather than return another start.
//      Anchors too long for a 16-bit half are scored here too, against whole strands; where even a 32-bit task cannot
//      hold the score (match * min(|anchor|, |read|) > 32767) the anchor gets no hit on that read and n_skipped counts it.
// Then the reference's rules, on the host.
#include "nr_batch.h"
#include "nr_launch_anchor.h"

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace {

constexpr int kMaxPairAnchor = (65535 - 65) / 4;   // a half holds 2 * score + 65 and score <= 2 * |anchor| (map-ont)
constexpr int kBufferLen = 100;                    // nanoRepeat_bam.py:221

inline char complement(char c) {
    switch (c) {
        case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A';
        case 'a': return 't'; case 'c': return 'g'; case 'g': return 'c'; case 't': return 'a';
        default: return c;
    }
}

// the smallest stripe height of the paired kernels that covers `rows` in as few stripes of at most 512 rows as possible
void pair_shape(int rows, int& R, int& S) {
    const int per_stripe = 32 * nr::pr::kMaxRPair2;
    S = std::max(1, (rows + per_stripe - 1) / per_stripe);
    const int need = (rows + 32 * S - 1) / (32 * S);
    R = nr::pr::kMaxRPair2;
    for (int h : {4, 6, 8, 12, 16})
        if (h >= need) { R = h; break; }
}

struct Cand { int score = 0, tstart = -1, tend = 0; };      // one anchor on one strand of one read

int anchor_regions(const nr_scoring_t* sc, int n_regions, const nr_anchor_region_t* regs, nr_anchor_read_t* out, nr_stats_t* stats) {
    // ---- reads of every region: split the lines, pack both strands ----
    std::vector<long long> first(n_regions + 1, 0);
    for (int g = 0; g < n_regions; ++g) {
        const nr_anchor_region_t& G = regs[g];
        if (G.n_reads < 0 || G.n_left < 0 || G.n_right < 0 || G.reads_len < 0 || (G.n_left > 0 && !G.left) ||
            (G.n_right > 0 && !G.right) || (G.n_reads > 0 && !G.reads))
            return nri::fail(NR_ERR_ARG, "nr_anchor_regions: a region has bad arguments");
        first[g + 1] = first[g] + G.n_reads;
    }
    const long long total = first[n_regions];
    std::vector<const char*> rptr(total);
    std::vector<int> rlen(total);
    for (int g = 0; g < n_regions; ++g) {
        const nr_anchor_region_t& G = regs[g];
        long long pos = 0, r = first[g];
        for (int i = 0; i < G.n_reads; ++i) {
            const char* nl = pos < G.reads_len ? static_cast<const char*>(memchr(G.reads + pos, '\n', (size_t)(G.reads_len - pos))) : nullptr;
            const long long end = nl ? nl - G.reads : G.reads_len;
            if ((!nl && i + 1 < G.n_reads) || (nl && i + 1 == G.n_reads) || end - pos > 0x7fffffffLL)
                return nri::fail(NR_ERR_BAD_BASE, "nr_anchor_regions: region %d does not hold %d lines (a read holds a newline?)", g, G.n_reads);
            rptr[r + i] = G.reads + pos;
            rlen[r + i] = (int)(end - pos);
            pos = end + 1;
        }
    }
    int rc = nri::ensure_init();
    if (rc) return rc;
    nr_stats_t st = {};
    nri::Pool pool;        // anchors are queries (an ambiguity plane for bases other than ACGT), read strands templates
    {
        size_t words = 0;
        for (long long i = 0; i < total; ++i) words += 2 * ((size_t)(rlen[i] + 15) / 16 + 1);
        pool.words.reserve(words + 4096);
    }
    std::vector<long long> left_word(n_regions, -1), right_word(n_regions, -1);
    for (int g = 0; g < n_regions; ++g) {
        left_word[g] = pool.add(regs[g].left, regs[g].n_left, true);
        right_word[g] = pool.add(regs[g].right, regs[g].n_right, true);
    }
    // per read: the words of its two strands (-1: not scored -- a base other than ACGT, empty, or over the template limit)
    std::vector<long long> fwd_word(total, -1), rev_word(total, -1);
    std::vector<std::string> rev(total);
    for (long long i = 0; i < total; ++i) {
        if (rlen[i] == 0) continue;
        if (rlen[i] > nrh::kMaxTlen) { ++st.n_skipped; continue; }
        const long long w = pool.add(rptr[i], rlen[i], false);
        if (w < 0) { ++st.n_skipped; continue; }
        fwd_word[i] = w;
        std::string& s = rev[i];
        s.resize(rlen[i]);
        for (int j = 0; j < rlen[i]; ++j) s[j] = complement(rptr[i][rlen[i] - 1 - j]);
        rev_word[i] = pool.add(s.data(), rlen[i], false);
    }
    if (pool.words.size() > 0xfffffff0ULL) return nri::fail(NR_ERR_TOO_LARGE, "nr_anchor_regions: sequence pool exceeds 2^32 words");

    // cand[(4 * read + 2 * anchor + strand)]: anchor 0 left, 1 right; strand 0 '+', 1 '-'
    std::vector<Cand> cand(4 * (size_t)total);

    // ---- launch 1: both anchors of a region per read strand on u16x2 words ----
    std::vector<nr::pr::AnchorPair> pairs;
    std::vector<long long> pair_slot;        // 4 * read + strand (the anchors' slots follow from it)
    int max_multi_t = 1;
    for (int g = 0; g < n_regions; ++g) {
        const nr_anchor_region_t& G = regs[g];
        const int qa = G.n_left <= kMaxPairAnchor ? G.n_left : 0, qb = G.n_right <= kMaxPairAnchor ? G.n_right : 0;
        int R = 0, S = 0;
        if (qa > 0 || qb > 0) pair_shape(std::max(qa, qb), R, S);
        for (long long i = first[g]; i < first[g + 1]; ++i) {
            if (fwd_word[i] < 0) continue;
            st.algorithmic_cells += 2LL * ((long long)G.n_left + G.n_right) * rlen[i];    // long anchors included
            for (int sd = 0; sd < 2 && S > 0; ++sd) {
                nr::pr::AnchorPair p = {};
                p.t_word = (uint32_t)(sd ? rev_word[i] : fwd_word[i]); p.t_len = rlen[i];
                p.qa_word = (uint32_t)left_word[g]; p.q_a = qa;
                p.qb_word = (uint32_t)right_word[g]; p.q_b = qb;
                p.R = R; p.S = S; p.out = (int)pairs.size();
                pairs.push_back(p);
                pair_slot.push_back(4 * i + sd);
                if (S > 1) max_multi_t = std::max(max_multi_t, rlen[i]);
                st.executed_cells += 2LL * 32 * R * S * rlen[i];
            }
        }
    }
    const int n_pairs = (int)pairs.size();
    if (n_pairs) {
        std::vector<nr::pr::AnchorPair> order(pairs);        // longest first: the launch's tail is made of short ones
        std::stable_sort(order.begin(), order.end(), [](const nr::pr::AnchorPair& x, const nr::pr::AnchorPair& y) {
            return (long long)x.R * x.S * x.t_len > (long long)y.R * y.S * y.t_len;
        });
        const int blocks = std::max(1, std::min(nri::sm_count(), (n_pairs + nr::kWarpsPerBlock - 1) / nr::kWarpsPerBlock));
        const size_t stride = (size_t)(max_multi_t + 31) / 32 * 32;
        const size_t pair_bytes = sizeof(nr::pr::AnchorPair) * n_pairs, pool_bytes = sizeof(uint32_t) * (pool.words.size() + 4),
                     key_bytes = sizeof(uint2) * n_pairs,
                     scratch_bytes = sizeof(ulonglong2) * 2 * stride * (size_t)blocks * nr::kWarpsPerBlock;
        nri::Bufs bufs;
        void *h_in = nullptr, *d_in = nullptr, *d_keys = nullptr, *h_keys = nullptr, *d_scratch = nullptr, *d_counter = nullptr;
        if ((rc = bufs.get(&h_in, pair_bytes + pool_bytes, true)) || (rc = bufs.get(&d_in, pair_bytes + pool_bytes, false)) ||
            (rc = bufs.get(&d_keys, key_bytes, false)) || (rc = bufs.get(&h_keys, key_bytes, true)) ||
            (rc = bufs.get(&d_scratch, scratch_bytes, false)) || (rc = bufs.get(&d_counter, 256, false)))
            return rc;
        memcpy(h_in, order.data(), pair_bytes);
        memcpy(static_cast<char*>(h_in) + pair_bytes, pool.words.data(), sizeof(uint32_t) * pool.words.size());
        cudaStream_t s = nri::stream();
        CUDA_TRY(cudaMemcpyAsync(d_in, h_in, pair_bytes + pool_bytes, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemsetAsync(d_counter, 0, 256, s));
        int* counter = static_cast<int*>(d_counter);
        CUDA_TRY(nrl::launch_anchor_pairs(blocks, s, static_cast<const nr::pr::AnchorPair*>(d_in), n_pairs,
                                      reinterpret_cast<const uint32_t*>(static_cast<char*>(d_in) + pair_bytes),
                                      static_cast<ulonglong2*>(d_scratch), stride, counter, static_cast<uint2*>(d_keys)));
        CUDA_TRY(cudaMemcpyAsync(h_keys, d_keys, key_bytes, cudaMemcpyDeviceToHost, s));
        int spin = 0;
        CUDA_TRY(cudaMemcpyAsync(&spin, counter + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        if (spin) return nri::fail(NR_ERR_CUDA, "nr_anchor_regions: a stripe gave up waiting for the stripe above it");
        ++st.kernel_launches;
        st.n_tasks += n_pairs;
        st.h2d_bytes += (int64_t)(pair_bytes + pool_bytes);
        st.d2h_bytes += (int64_t)key_bytes;
        const uint2* keys = static_cast<const uint2*>(h_keys);
        for (int p = 0; p < n_pairs; ++p) {
            const long long slot = pair_slot[p];
            const long long i = slot / 4;
            const int sd = (int)(slot % 4);
            const unsigned k2[2] = {keys[p].x, keys[p].y};
            for (int a = 0; a < 2; ++a) {
                if ((a ? pairs[p].q_b : pairs[p].q_a) == 0 || k2[a] == 0) continue;
                Cand& c = cand[4 * i + 2 * a + sd];
                c.score = (int)(k2[a] >> 17);
                c.tend = 0xffff - (int)((k2[a] >> 1) & 0xffffu) + 1;
            }
        }
    }

    // ---- the rules of nanoRepeat_bam.py:165-179 on one anchor's two candidates ----
    const int min_score = std::max(1, sc->min_dp_score);
    auto hits_of = [&](long long i, int a, int* idx) {          // -> number of hits; idx: strands, best first ('+' on a tie)
        int n = 0;
        for (int sd = 0; sd < 2; ++sd) {
            const Cand& c = cand[4 * i + 2 * a + sd];
            if (c.score > 0 && c.score >= min_score) idx[n++] = sd;
        }
        if (n == 2 && cand[4 * i + 2 * a + 1].score > cand[4 * i + 2 * a].score) std::swap(idx[0], idx[1]);
        return n;
    };
    // hits[0].align_len < 10 (:173) cannot happen: a hit scores >= min_dp_score >= 10 * match, so it spans >= 10 read bases;
    // mapq > 30 is taken as true (anchoring.py)
    auto good = [&](long long i, int a, const int* idx, int n) {
        if (n == 0) return false;
        if (n == 1) return true;
        return 2LL * cand[4 * i + 2 * a + idx[0]].score > 3LL * cand[4 * i + 2 * a + idx[1]].score;     // AS0 > 1.5 * AS1
    };

    // ---- launch 2: start columns (windows of the good anchors' best hits) and anchors too long for a half ----
    std::vector<const char*> tq, tt;
    std::vector<int32_t> tql, ttl;
    std::vector<long long> tslot;           // candidate slot the task fills
    std::vector<int> twin;                  // window start a (-1: a whole strand)
    const int min_open = std::min(sc->gap_open1, sc->gap_open2), min_ext = std::min(sc->gap_ext1, sc->gap_ext2);
    for (int g = 0; g < n_regions; ++g) {
        const nr_anchor_region_t& G = regs[g];
        for (int a = 0; a < 2; ++a) {
            const int n = a ? G.n_right : G.n_left;
            const char* q = a ? G.right : G.left;
            for (long long i = first[g]; i < first[g + 1]; ++i) {
                if (fwd_word[i] < 0 || n == 0) continue;
                if (n > kMaxPairAnchor) {
                    if ((long long)sc->match * std::min(n, rlen[i]) > nri::kMaxScore) {     // no DP word holds its score:
                        ++st.n_skipped;                                                     // no hit, counted once
                        continue;
                    }
                    for (int sd = 0; sd < 2; ++sd) {
                        tq.push_back(q); tql.push_back(n);
                        tt.push_back(sd ? rev[i].data() : rptr[i]); ttl.push_back(rlen[i]);
                        tslot.push_back(4 * i + 2 * a + sd); twin.push_back(-1);
                    }
                    continue;
                }
                int idx[2];
                const int nh = hits_of(i, a, idx);
                if (!good(i, a, idx, nh)) continue;
                const Cand& c = cand[4 * i + 2 * a + idx[0]];
                const long long W = n + std::max(0LL, ((long long)sc->match * n - c.score - min_open) / min_ext);
                const int w0 = (int)std::max(0LL, (long long)c.tend - W);
                tq.push_back(q); tql.push_back(n);
                tt.push_back((idx[0] ? rev[i].data() : rptr[i]) + w0); ttl.push_back(c.tend - w0);
                tslot.push_back(4 * i + 2 * a + idx[0]); twin.push_back(w0);
            }
        }
    }
    if (!tq.empty()) {
        const int nt = (int)tq.size();
        nr_batch_t* b = nr_batch_create_tasks(sc, nt, tq.data(), tql.data(), tt.data(), ttl.data());
        if (!b) return nri::last_code();
        std::vector<nr_aln_t> res(nt);
        rc = nr_batch_run(b, nullptr);
        if (!rc) rc = nr_batch_fetch_alns(b, res.data());
        nr_stats_t bs = {};
        if (!rc) rc = nr_batch_stats(b, &bs);
        nr_batch_destroy(b);
        if (rc) return rc;
        st.executed_cells += bs.executed_cells; st.n_tasks += bs.n_tasks; st.kernel_launches += bs.kernel_launches;
        st.n_skipped += bs.n_skipped; st.h2d_bytes += bs.h2d_bytes; st.d2h_bytes += bs.d2h_bytes;
        for (int t = 0; t < nt; ++t) {
            Cand& c = cand[tslot[t]];
            if (twin[t] < 0) {             // a whole strand (long anchor): the record as it is (tstart kept for good anchors)
                c.score = res[t].score; c.tstart = res[t].tstart; c.tend = res[t].tend;
                continue;
            }
            if (res[t].score != c.score || res[t].tend != c.tend - twin[t])
                return nri::fail(NR_ERR_CUDA, "nr_anchor_regions: start recovery of a hit (%d, end %d) found (%d, %d, %d) in its window",
                                 c.score, c.tend, res[t].score, twin[t] + res[t].tstart, twin[t] + res[t].tend);
            c.tstart = twin[t] + res[t].tstart;
        }
    }

    // ---- acceptance, distance, core and middle positions (nanoRepeat_bam.py:181-234) ----
    for (long long i = 0; i < total; ++i) {
        nr_anchor_read_t& o = out[i];
        memset(&o, 0, sizeof o);
        o.read_len = rlen[i];
        int idx[2][2], nh[2];
        nr_aln_t* best[2] = {&o.left, &o.right};
        uint8_t* strand[2] = {&o.left_strand, &o.right_strand};
        bool ok[2];
        for (int a = 0; a < 2; ++a) {
            nh[a] = hits_of(i, a, idx[a]);
            ok[a] = good(i, a, idx[a], nh[a]);
            best[a]->tstart = -1;
            if (nh[a]) {
                const Cand& c = cand[4 * i + 2 * a + idx[a][0]];
                best[a]->score = c.score; best[a]->tend = c.tend;
                if (ok[a]) best[a]->tstart = c.tstart;                    // whole-strand records carry one either way
                *strand[a] = idx[a][0] ? '-' : '+';
            }
        }
        o.left_good = ok[0]; o.right_good = ok[1];
        if (!ok[0] || !ok[1]) continue;
        const int dist = o.left_strand == o.right_strand ? o.right.tstart - o.left.tend : 0;          // :204-207
        o.dist_between_anchors = dist;
        if (!(dist > -10)) continue;                                                                  // :209-211
        o.accepted = 1;
        o.strand = o.left_strand;
        o.mid_start = o.left.tend;                                                                    // :221-234
        o.mid_end = o.right.tstart;
        o.core_start = std::max(o.left.tend - kBufferLen, 0);
        o.core_end = std::min(o.right.tstart + kBufferLen, rlen[i]);
        o.left_buffer = o.left.tend - o.core_start;
        o.right_buffer = o.core_end - o.right.tstart;
    }
    if (stats) *stats = st;
    return NR_OK;
}

}  // namespace

extern "C" int nr_anchor_regions(const nr_scoring_t* sc, int32_t n_regions, const nr_anchor_region_t* regions, nr_anchor_read_t* out,
                                 nr_stats_t* stats) {
    if (nri::check(sc)) return nri::last_code();
    if (n_regions < 0 || (n_regions > 0 && !regions)) return nri::fail(NR_ERR_ARG, "nr_anchor_regions: bad arguments");
    if (!nrh::is_map_ont(*sc) || sc->min_dp_score < 10 * sc->match)
        return nri::fail(NR_ERR_ARG, "nr_anchor_regions: needs map-ont scoring with min_dp_score >= 10 * match");
    long long total = 0;
    for (int g = 0; g < n_regions; ++g) total += std::max(0, regions[g].n_reads);
    if (total > 0 && !out) return nri::fail(NR_ERR_ARG, "nr_anchor_regions: out is NULL");
    return anchor_regions(sc, n_regions, regions, out, stats);
}
