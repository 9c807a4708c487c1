// nr_window_kernel.cuh -- the joint path's alignment: best local alignment AND the score of that alignment inside a
// window of the template, in one DP (no traceback, no CIGAR).
//
// nanoRepeat-joint (reference src/NanoRepeat/nanoRepeat_joint.py:275-343, :376-419) aligns every read against a grid of
// templates  left + motif1*k1 + mid + motif2*k2 + right  with minimap2 -c --eqx and then RE-SCORES the CIGAR inside the
// window [|left| - 10, |left| + m1 k1 + |mid| + m2 k2 + 10) with tk.target_region_alignment_stats_from_cigar
// (tk.py:435-500): +2 per '=', -4 per 'X', a deletion by the part of it inside the window (-4 - 2 (part - 1)), an
// insertion in full (-4 - 2 (len - 1)) when its template position p satisfies a < p < b - 1.  Per read the grid point
// with the best window score wins (nanoRepeat_joint.py:457-476).
//
// What the device returns per (read, template) is therefore two integers, the alignment score and the window score of
// the optimal path.  DP word:  w = score * 65536 + payload,  payload = window score collected so far.  Every move adds
// its alignment score to the upper half and, when it lies in the window, its re-scoring value to the lower half:
//   diagonal into template position p:            +2 / -4 (match / mismatch) if a <= p < b
//   deletion step consuming template position p:  -4 if it opens the run or p == a, else -2, if a <= p < b
//   insertion step at template position p:        -4 if it opens the run, else -2, if a < p < b - 1
// Integer max on words is the lexicographic max of (score, payload): among all optimal alignments the canonical one is
// the one with the highest window score (the CPU checker under oracle/ has the same rule and a traceback; the
// golden vectors run the reference's own CIGAR re-scoring on the traceback's CIGAR).  Score range: the payload decodes
// as a signed 16-bit value.  Its ceiling is +2 per window base, +16 000 at the 8 000-base window limit.  Its floor is an
// insertion charged in full, bounded by the score limit (match * min(q, t) <= 32 767): a 16 356-base insertion into a
// 3-base window of a 16 383-base template gives (16 386, -32 708), 60 from the decode limit at the score limit
// (tests/test_gpu_joint_edges.py).
//
// Mapping: one warp per (read, template) task, 8 rows per lane, the read cut into stripes of 256 rows that the SAME warp
// sweeps one after the other; the bottom row of a stripe (H, F1, F2 per template column) travels through a per-warp
// scratch row in global memory (L2), read back 32 columns at a time.  The wavefront is skewed (lane l works on column
// step - l) and the bottom row moves down the lanes by shuffle, as in nr_kernels.cuh.
#pragma once
#include "nr_launch_window.h"
#include <type_traits>

namespace nrw {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kPad = -(16384 << 16);

__device__ __forceinline__ bool amb_base(const uint32_t* __restrict__ q, uint32_t plane, int i) {
    return plane && ((q[plane + (i >> 5)] >> (i & 31)) & 1u);
}

// Substitution words of one stripe: prof[(win * 4 + c) * kRows + lane * kR + r], c = template code, win = 1 inside the window.
__device__ __forceinline__ void build_profile(int* prof, const uint32_t* __restrict__ q, int q_len, bool reverse, int row0,
                                              int lane, const WinScore& sc) {
    const uint32_t plane = q[(q_len + 15) >> 4];
#pragma unroll
    for (int r = 0; r < kR; ++r) {
        const int i = row0 + lane * kR + r;
        int code = 4;
        if (i < q_len) {
            const int qi = reverse ? q_len - 1 - i : i;
            code = (q[qi >> 4] >> (30 - 2 * (qi & 15))) & 3;
            if (reverse) code ^= 2;      // complement under the packer's codes A0 C1 T2 G3: A<->T, C<->G
            if (amb_base(q, plane, qi)) code = 5;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int out = code == 4 ? kPad : code == 5 ? sc.ambiguous : (code == c ? sc.match : sc.mismatch);
            const int pay = code == 4 ? 0 : (code == c ? 2 : -4);                      // '=' +2, 'X' -4 (tk.py:444-445)
            prof[(c) * kRows + lane * kR + r] = out;
            prof[(4 + c) * kRows + lane * kR + r] = out + pay;
        }
    }
}

// One task.  bnd: two rows of int4 per template column (ping-pong between consecutive stripes).
__device__ __forceinline__ int window_task(const WinTask& tk, const uint32_t* __restrict__ pool, const WinScore& sc, int* prof,
                                           int4* bnd, int lane) {
    const uint32_t* q = pool + tk.q_word;
    const uint32_t* tw = pool + tk.t_word;
    const int t_len = tk.t_len, a = tk.win_a, b = tk.win_b;
    const int n_stripes = (tk.q_len + kRows - 1) / kRows;
    int best = 0;
    for (int s = 0; s < n_stripes; ++s) {
        __syncwarp();
        build_profile(prof, q, tk.q_len, tk.reverse != 0, s * kRows, lane, sc);
        __syncwarp();
        const int4* bin = bnd + (size_t)((s + 1) & 1) * t_len;      // written by stripe s - 1
        int4* bout = bnd + (size_t)(s & 1) * t_len;
        const bool top = s > 0, bot = s + 1 < n_stripes;
        int H[kR], E1[kR], E2[kR];
#pragma unroll
        for (int r = 0; r < kR; ++r) { H[r] = 0; E1[r] = sc.open1; E2[r] = sc.open2; }
        // (E of column 0 -> 1: a gap that opens at template position 0; its window value is added when it is used below)
        int hup_prev = 0, h_out = 0, f1_out = 0, f2_out = 0;
        int4 bcur = make_int4(0, 0, 0, 0);
        const int nsteps = t_len + 31;
        // one column step of this lane; GUARD: the lane may be outside the matrix (the first 31 and the last 31 steps)
        auto step = [&](int st, auto guard_tag) {
            constexpr bool GUARD = decltype(guard_tag)::value;
            if (top && (st & 31) == 0) {
                const int cj = st + lane;
                bcur = cj < t_len ? __ldcg(&bin[cj]) : make_int4(0, 0, 0, 0);
            }
            int hup = __shfl_up_sync(kFull, h_out, 1);
            int f1 = __shfl_up_sync(kFull, f1_out, 1);
            int f2 = __shfl_up_sync(kFull, f2_out, 1);
            if (top) {        // (uniform)
                const int bh = __shfl_sync(kFull, bcur.x, st & 31), bf1 = __shfl_sync(kFull, bcur.y, st & 31), bf2 = __shfl_sync(kFull, bcur.z, st & 31);
                if (lane == 0) { hup = bh; f1 = bf1; f2 = bf2; }
            } else if (lane == 0) { hup = 0; f1 = kPad; f2 = kPad; }
            const int p = st - lane;                 // template position of this lane's column
            if (!GUARD || (p >= 0 && p < t_len)) {
                const int code = (tw[p >> 4] >> (30 - 2 * (p & 15))) & 3;
                const bool in_diag = p >= a && p < b;                 // this column's base is inside the window
                const bool in_next = p + 1 >= a && p + 1 < b;         // the next column's (a deletion step computed here consumes it)
                const bool in_ins = p + 1 > a && p + 1 < b - 1;       // insertions behind this column (tk.py:477)
                const int h_open_pay = in_next ? -4 : 0, h_ext_pay = in_next ? (p + 1 == a ? -4 : -2) : 0;
                const int v_open_pay = in_ins ? -4 : 0, v_ext_pay = in_ins ? -2 : 0;
                const int ho1 = sc.open1 + h_open_pay, ho2 = sc.open2 + h_open_pay, he1 = sc.ext1 + h_ext_pay, he2 = sc.ext2 + h_ext_pay;
                const int vo1 = sc.open1 + v_open_pay, vo2 = sc.open2 + v_open_pay, ve1 = sc.ext1 + v_ext_pay, ve2 = sc.ext2 + v_ext_pay;
                const int4* pr = reinterpret_cast<const int4*>(prof + ((in_diag ? 4 : 0) + code) * kRows + lane * kR);
                int hd = hup_prev;
                hup_prev = hup;
                int cm = best;
#pragma unroll
                for (int c = 0; c < kR / 4; ++c) {
                    const int4 sv = pr[c];
                    const int s4[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int r = 4 * c + u;
                        const int hleft = H[r];
                        const int t = __vimax3_s32(hd + s4[u], E1[r], E2[r]);
                        const int h = __vimax3_s32_relu(t, f1, f2);
                        E1[r] = __viaddmax_s32(h, ho1, E1[r] + he1);
                        E2[r] = __viaddmax_s32(h, ho2, E2[r] + he2);
                        f1 = __viaddmax_s32(h, vo1, f1 + ve1);
                        f2 = __viaddmax_s32(h, vo2, f2 + ve2);
                        hd = hleft;
                        H[r] = h;
                        if (r & 1) cm = __vimax3_s32(cm, h, H[r - 1]);
                    }
                }
                best = cm;
                h_out = H[kR - 1]; f1_out = f1; f2_out = f2;
                if (bot && lane == 31) __stcg(&bout[p], make_int4(h_out, f1_out, f2_out, 0));
            }
        };
        int st = 0;
        for (; st < min(31, nsteps); ++st) step(st, std::true_type{});
#pragma unroll 2
        for (; st < t_len; ++st) step(st, std::false_type{});          // every lane's column is inside the matrix
        for (; st < nsteps; ++st) step(st, std::true_type{});
        __syncwarp();
        __threadfence_block();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(kFull, best, o));
    return best;
}

// out[task] = (alignment score, window score of the canonical optimal alignment)
__global__ void __launch_bounds__(32 * kWarps)
window_kernel(const WinTask* __restrict__ tasks, int n_tasks, const uint32_t* __restrict__ pool, WinScore sc, int4* scratch,
              int scratch_stride, int* counter, int2* out) {
    extern __shared__ int wsmem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int* prof = wsmem + warp * (8 * kRows);
    int4* bnd = scratch + (size_t)(blockIdx.x * kWarps + warp) * scratch_stride;
    for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(counter, 1);
        i = __shfl_sync(kFull, i, 0);
        if (i >= n_tasks) break;
        const WinTask tk = tasks[i];
        int w = 0;
        if (tk.q_len > 0 && tk.t_len > 0) w = window_task(tk, pool, sc, prof, bnd, lane);
        if (lane == 0) {
            const int score = (w + 0x8000) >> 16;                  // payload is a signed 16-bit value around the score field
            out[i] = make_int2(score, w - (score << 16));
        }
    }
}

}  // namespace nrw
