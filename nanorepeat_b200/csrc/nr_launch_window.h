// nr_launch_window.h -- the joint path's kernels (nr_launch_window.cu: nr_window_kernel.cuh, nr_window_ladder.cuh) as
// the host side (nr_joint.cu) sees them: the task records, the scoring words and one launcher per kernel.  Every
// launcher sets its kernel's maximum dynamic shared memory once and returns the launch's cudaError_t.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace nrw {

struct WinTask {           // 32 bytes
    uint32_t q_word;       // 2-bit packed read (same pool layout as nr_kernels.cuh, ambiguity plane included)
    int32_t  q_len;
    uint32_t t_word;       // 2-bit packed template
    int32_t  t_len;
    int32_t  win_a, win_b; // window [a, b) in template coordinates
    int32_t  reverse;      // 1: align the reverse complement of the read
    int32_t  pad;
};

constexpr int kR = 8;                  // rows per lane
constexpr int kRows = 32 * kR;         // rows per stripe
constexpr int kWarps = 8;              // warps per block

struct WinScore {          // scoring as word increments (upper half: alignment score)
    int match, mismatch, ambiguous;          // a << 16, -(b << 16), -(sc_ambi << 16)
    int open1, ext1, open2, ext2;            // -((q + e) << 16), -(e << 16), ...
};

struct LadBwdTask {        // one per (read, strand)
    uint32_t q_word; int32_t q_len;
    uint32_t rev_word; int32_t n_right;    // reverse(right)
    int32_t reverse;                       // strand
    int32_t pad;
    // First word of this task's junction vectors (3 planes of q_len words).  64-bit: a call spends 6 words per read base
    // on the shared path, past 2^31 after ~358 M bases.  Kept as two 32-bit halves: a long long member makes the struct
    // 8-byte aligned, and ptxas then gives both ladder kernels 128 registers (64 / 80 with the halves) and a spill.
    uint32_t bvec_lo, bvec_hi;
    __host__ __device__ long long bvec_off() const { return (long long)(((unsigned long long)bvec_hi << 32) | bvec_lo); }
    void set_bvec_off(long long w) { bvec_lo = (uint32_t)w; bvec_hi = (uint32_t)((unsigned long long)w >> 32); }
};
static_assert(sizeof(LadBwdTask) == 32, "LadBwdTask is 32 bytes");

struct LadFwdTask {        // one per (read, strand, k1)
    uint32_t q_word; int32_t q_len;
    uint32_t t_word;                       // left + motif1*k1 + mid + motif2*k2max(of the locus)
    int32_t n_pre;                         // |left| + m1*k1 + |mid|: columns before the second repeat
    int32_t m2, k2_first, k2_step, k2_count;
    int32_t win_a;                         // |left| - 10 (>= 0)
    int32_t reverse;
    int32_t bwd;                           // index of the (read, strand)'s LadBwdTask
    int32_t out_off;                       // first record of this task in out[]: k2_count records (prefix: in pbest1[])
    int32_t mode;                          // kWhole / kPrefix / kCont
    int32_t pbest1;                        // kCont: index into pbest1[] of this k1's entry
    long long cstate;                      // kPrefix: first word of its saved columns [k][3][q_len]; kCont: of its own column
};
// kWhole: the whole forward template from the empty column.  kPrefix: the fields n_pre / m2 / k2_* describe the k1
// junctions (n_pre = |left|, m2 = m1, ...); nothing is joined, states are saved.  kCont: t_word = mid + motif2*k2max,
// n_pre = |mid|, every column inside the window.
constexpr int kWhole = 0, kPrefix = 1, kCont = 2;

constexpr int kMaxK2 = 64;                 // grid points per forward task (shared-memory tables)

}  // namespace nrw

namespace nrl {
// 32 * kWarps threads a block; scratch: scratch_stride int4 per warp of the launch; counter: zeroed work counter
cudaError_t launch_window(int blocks, cudaStream_t st, const nrw::WinTask* tasks, int n_tasks, const uint32_t* pool,
                          const nrw::WinScore& sc, int4* scratch, int scratch_stride, int* counter, int2* out);
cudaError_t launch_ladder_bwd(int blocks, cudaStream_t st, const nrw::LadBwdTask* tasks, int n_tasks, const uint32_t* pool,
                              const nrw::WinScore& sc, int4* scratch, int scratch_stride, int* counter, int* bvec, int* ronly);
cudaError_t launch_ladder_fwd(int blocks, cudaStream_t st, const nrw::LadFwdTask* tasks, int n_tasks, const nrw::LadBwdTask* btasks,
                              const uint32_t* pool, const nrw::WinScore& sc, int4* scratch, int scratch_stride, int* counter,
                              const int* bvec, const int* ronly, int* cstate, int* pbest1, int2* out);
}  // namespace nrl
