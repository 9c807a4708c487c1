// nr_batch.h -- the batch behind the C ABI's nr_batch_t and the host services its planner (nr_plan.cu) shares with
// nr_api.cu and nr_anchor.cu.  Host-only translation units include it; kernel translation units must not (their code
// placement follows the exact text they are compiled from, DESIGN.md sections 4.10 and 9).
#pragma once
#include "nr_internal.h"
#include "nr_launch.h"

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <string>
#include <thread>
#include <vector>

namespace nrh {

constexpr int kMaxScore = 32767;   // signed 16-bit score field of the packed DP word
constexpr int kMaxTlen = 65535 - 64; // unsigned 16-bit span field, minus the wavefront skew (step counters share it)

int fail(int code, const char* fmt, ...);     // records the thread's last error (nr_last_error), returns code

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
        if (!nri::pack(s, len, words.data() + w0)) {
            if (!ambiguous_ok) { words.resize(w0); return -1; }
            link_plane(w0, s, len);
        }
        return (long long)w0;
    }
    // append the ambiguity plane of the read packed at word w0 and link it from the read's slack word
    void link_plane(size_t w0, const char* s, int len) {
        const size_t at = words.size();
        words.resize(at + (size_t)(len + 31) / 32, 0u);
        nri::ambiguity(s, len, words.data() + at);
        words[w0 + (size_t)(len + 15) / 16] = (uint32_t)(at - w0);
    }
};

struct Launch {      // one persistent launch per batch
    bool ladder;     // ladder_kernel over nr_batch::ltasks instead of exact_kernel over nr_batch::tasks
    int R;           // tallest stripe of the launch: sizes the shared memory per warp
    int count;
    int blocks;
    bool fixed;      // scoring == map-ont: kernels with immediate constants
    // paired launch (nr_pair_kernels.cuh): two reads of one region per warp
    int n_pairs;
    int pair_R;
    int pair_blocks;
    int redo_R;                 // tallest stripe among the paired round-3 reads: sizes the redo launch
};

struct RegionInfo {   // one add_round2 / add_round3 call
    int n_left = 0, n_right = 0, motif_len = 0;
    int first_read = 0, n_reads = 0;
    std::string left, motif;      // round 2 keeps them for a round-3 batch built over the same reads
};

// The uploaded blob: sections at 256-byte boundaries in this order, then 256 bytes of counters (zeroed)
enum BlobSection { SEC_TASKS, SEC_LREGS, SEC_ORDER, SEC_PAIRS, SEC_COOP, SEC_COOP_IDX, SEC_POOL, kBlobSections };
struct Section {
    const void* src;      // `bytes` bytes from here, then `zeros` zero bytes
    size_t bytes, zeros;
    size_t off;           // in the blob
};

enum BatchKind { KIND_TASKS = 0, KIND_ROUND2 = NR_KIND_ROUND2, KIND_ROUND3 = NR_KIND_ROUND3 };

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

inline bool is_map_ont(const nr_scoring_t& c) {
    return c.match == 2 && c.mismatch == 4 && c.gap_open1 == 4 && c.gap_ext1 == 2 && c.gap_open2 == 24 && c.gap_ext2 == 1 &&
           c.ambiguous == 1;
}

// NR_TRACE=1: host-side phase times of a commit on stderr (where a commit's half millisecond goes)
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

}  // namespace nrh

struct nr_batch {
    nrh::BatchKind kind = nrh::KIND_TASKS;
    nr_scoring_t sc = {};
    bool committed = false;
    std::vector<nr::Task> tasks;
    std::vector<nr::LadderTask> ltasks;       // round 3 in ladder mode (tasks stays empty)
    std::vector<nr::LadderRegion> lregs;
    bool ladder = false;
    bool flag = false;                        // ladder on flag words: d_out holds (score, spans both, ends in right)
    bool pair = false;                        // paired u16x2 kernels where a task is eligible (round 2: flags kind; round 3: mode 3)
    bool r2flags = false;                     // round 2: records are (score, span predicate, tend); no tstart
    std::vector<nr::pr::Pair2> pairs2;        // single-stripe pairs first (n_pairs2_single), then the pairs of long reads
    std::vector<nr::pr::Pair3> pairs3;
    int n_pairs2_single = 0, n_pairs3_single = 0;
    bool long_redone = false;                 // the host-side rescoring of this run's undecidable long reads is merged
    int n_long_pairs = 0;                     // pairs of long reads: their stripes are entries of order[] (nr::pr::kPairEntry)
    void* d_pairs = nullptr;                  // inside the blob
    uint2* d_prung = nullptr;                 // round 3 pairs: (P, J) tokens per rung of a pair's ladder
    size_t prung_bytes = 0;
    int32_t* d_redo = nullptr;                // round 3 pairs: reads to rescore on 32-bit flag words
    size_t redo_bytes = 0;
    cudaEvent_t ev_t[6] = {};                 // nr_set_timing(1): start / end of the 32-bit, paired and redo launches
    bool timed[3] = {};
    int* h_redo_count = nullptr;              // pinned
    int* h_spin = nullptr;                    // pinned: the kernels' give-up flag after the run (long reads only)
    long long paired_cells = 0, rest_cells = 0;
    long long paired_useful = 0, rest_useful = 0;   // the same without padding: rows of real reads only
    bool round2_exit = false;                 // the single-stripe round-2 pairs may end their sweeps early (Pair2::check_col)
    size_t n_out = 0;                         // records in d_out / h_out
    std::vector<int32_t> order;               // entries of the 32-bit launch: (task << 7) | code (nr_kernels.cuh)
    std::vector<nr::CoopInfo> coop;           // scratch of the multi-stripe tasks
    std::vector<int32_t> coop_idx;            // exact tasks: index into coop, -1 for single-stripe tasks
    nr::CoopInfo* d_coop = nullptr;
    int32_t* d_coop_idx = nullptr;
    std::vector<int32_t> lt_src;              // round 3 over a round-2 batch's reads: that batch's task of every ladder task
    uint32_t* d_state = nullptr;              // round 2 pairs: DP state after column |left| - 2, kept for round 3
    uint32_t* d_kept = nullptr;               // round 2 dominance exit: 128 words per warp of the launch
    size_t state_bytes = 0;
    int* d_flags = nullptr;                   // progress flags of the multi-stripe tasks, zeroed before every run
    size_t flags_bytes = 0;
    nrh::Launch launch = {};
    nrh::Pool pool;
    // per-read bookkeeping (rounds 2 and 3)
    std::vector<nrh::RegionInfo> regions;
    int n_reads = 0;
    int n_skipped = 0;                        // tasks / reads left unscored (template not ACGT, beyond the packed range)
    int n_ambiguous_reads = 0;                // reads with a base other than ACGT (scored through an ambiguity plane)
    std::vector<int32_t> read_region;
    std::vector<int32_t> kmin, kmax;
    std::vector<int64_t> rung_off;            // n_reads + 1 (round 3)
    // device
    nrh::Section blob[nrh::kBlobSections] = {};   // layout of d_blob / h_blob (the counters follow the last section)
    void* d_blob = nullptr;                   // tasks | regions | order | pairs | coop | coop_idx | pool | counters: one H2D copy
    size_t blob_bytes = 0;
    void* h_blob = nullptr;                   // pinned staging of the same layout
    nr::Task* d_tasks = nullptr;
    nr::LadderTask* d_ltasks = nullptr;
    nr::LadderRegion* d_lregs = nullptr;
    int32_t* d_order = nullptr;
    uint32_t* d_pool = nullptr;
    int* d_counters = nullptr;
    int4* d_out = nullptr;
    size_t out_bytes = 0;
    int4* d_scratch = nullptr;
    size_t scratch_bytes = 0;
    int4* h_out = nullptr;                    // pinned
    int4* d_sel = nullptr;                    // flag ladder: per read (top score, n tied, sum k lo, sum k hi)
    int4* h_sel = nullptr;                    // pinned
    size_t sel_bytes = 0;
    nr_stats_t stats = {};
    bool ran = false;
    cudaStream_t run_stream = nullptr;        // stream of the last nr_batch_run: fetch orders itself behind it
    cudaEvent_t ev_uploaded = nullptr;        // recorded behind the upload on the library's stream
    cudaEvent_t ev_done = nullptr;            // recorded behind the kernel and the result copy of nr_batch_run
    int refs = 1;                             // the owner + round-3 batches that read this batch's packed reads
    nr_batch* qsrc = nullptr;                 // round 3: the committed round-2 batch whose reads are reused
};

namespace nrh {
// Plans a batch for a device with sm_count SMs (nr_plan.cu): pairs, stripe heights, the 32-bit launch's entries, buffer
// sizes and the blob's sections.  No CUDA call; nr_api.cu's upload_batch allocates and uploads what it decided.
int plan_batch(nr_batch* b, int sm_count);
}  // namespace nrh
