// nr_window_ladder.cuh -- the joint path with shared sweeps: nanoRepeat-joint's grid of templates
//     left + motif1*k1 + mid + motif2*k2 + right          (reference nanoRepeat_joint.py:351-374, grids :296-333, :397-410)
// scored for one read without sweeping every grid point's rectangle (nr_window_kernel.cuh does that and is the checker
// of this file in the tests).  Same DP word (score * 65536 + payload, payload = window score collected along the path)
// and the same contract: per grid point the best (score, payload), payload highest among the alignments of that score.
//
// What is shared.  For a fixed k1 the templates of all k2 have the prefix  left + motif1*k1 + mid + motif2*k2  and the
// suffix  right  in common, so -- exactly like the 1-D ladder of nr_kernels.cuh --
//   * ONE backward sweep per (read, strand): reversed read x reversed right.  Its last column gives, per read row, the
//     best continuation into the right anchor (junction vectors H, E1, E2); its running maximum is the class of
//     alignments that lie inside the right anchor alone;
//   * ONE forward sweep per (read, strand, k1) over left + motif1*k1 + mid + motif2*k2max.  Whenever a lane finishes a
//     junction column  n_pre + m2*k2  it joins its forward states with the junction vectors row by row; the maximum over
//     the rows (all stripes) is the class of alignments that cross the junction, the running maximum at that moment the
//     class of alignments that end before it.  Grid point (k1, k2) = the maximum of the three classes.
// Cells per read and strand:  |read| x (|right| + |K1| x (|left| + m1 k1 + |mid| + m2 k2max))  instead of
// |K1| |K2| x |read| x |template|: a factor |K2| / (1 + 1/|K1|), 5-6 on the coarse grids of round 2, 3-4 on round 3's.
//
// Sharing over k1 as well (the 2-D ladder).  The forward sweeps of all k1 have  left + motif1*k1  in common up to the
// column where motif1 stops, so when a read's K1 is an arithmetic progression too:
//   * ONE prefix sweep per (read, strand) over left + motif1*k1max.  Whenever a lane finishes the column before
//     c1(k1) = |left| + m1*k1 it saves its rows' states (H and the two gap states entering the next column) and the
//     running maximum: the DP column every template of that k1 continues from;
//   * per (read, strand, k1) ONE continuation sweep over  mid + motif2*k2max  that starts from the saved column instead
//     of the empty one, with the junctions per k2 as above.
// Cells per read and strand:  |read| x (|right| + |left| + m1 k1max + |K1| x (|mid| + m2 k2max)).
//
// The window and the payload across the junction.  The window of grid point (k1, k2) is [|left| - 10, J + 10) with J the
// junction column: in the forward sweep every column from |left| - 10 on is inside it for every k2; in the backward sweep
// the first ten bases of the right anchor are.  A deletion's window value depends only on how many of its bases lie in
// the window (-4 - 2 (n - 1), tk.py:484-488), so the backward sweep may charge it in its own direction (-4 at the first
// base it meets inside the window, -2 after); a deletion that SPANS the junction has bases inside the window on both
// sides and was opened twice, so its join gets the alignment's gap-open refund and +2 of payload.  An insertion's value
// depends only on its length and position, whichever way the rows are walked.
#pragma once
#include "nr_window_kernel.cuh"

namespace nrw {

// Substitution words of one stripe for the oriented read (strand: reverse complement), optionally walked backwards
// (backward sweep).  prof[(win * 4 + c) * kRows + lane * kR + r].
__device__ __forceinline__ void build_profile2(int* prof, const uint32_t* __restrict__ q, int q_len, bool strand, bool backwards,
                                               int row0, int lane, const WinScore& sc) {
    const uint32_t plane = q[(q_len + 15) >> 4];
#pragma unroll
    for (int r = 0; r < kR; ++r) {
        const int i = row0 + lane * kR + r;
        int code = 4;
        if (i < q_len) {
            const int j = backwards ? q_len - 1 - i : i;          // row of the oriented read
            const int qi = strand ? q_len - 1 - j : j;            // base of the read as stored
            code = (q[qi >> 4] >> (30 - 2 * (qi & 15))) & 3;
            if (strand) code ^= 2;
            if (amb_base(q, plane, qi)) code = 5;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int out = code == 4 ? kPad : code == 5 ? sc.ambiguous : (code == c ? sc.match : sc.mismatch);
            const int pay = code == 4 ? 0 : (code == c ? 2 : -4);
            prof[(c) * kRows + lane * kR + r] = out;
            prof[(4 + c) * kRows + lane * kR + r] = out + pay;
        }
    }
}

// ---- backward sweep: reversed oriented read x reverse(right) -------------------------------------------------------
// bvec[0 / 1 / 2][forward row i] = H / E1 + refund / E2 + refund of reversed row q - 2 - i in the last column; forward
// row q - 1 keeps (0, none, none): nothing of the read is left for the right anchor.  *ronly = best word of the sweep.
__device__ __forceinline__ void ladder_bwd_task(const LadBwdTask& tk, const uint32_t* __restrict__ pool, const WinScore& sc,
                                                int* prof, int4* bnd, int* bvec, int* ronly, int lane) {
    const uint32_t* q = pool + tk.q_word;
    const uint32_t* tw = pool + tk.rev_word;
    const int t_len = tk.n_right, q_len = tk.q_len;
    const int n_stripes = (q_len + kRows - 1) / kRows;
    const int refund1 = -sc.open1 + sc.ext1 + 2, refund2 = -sc.open2 + sc.ext2 + 2;      // gap open (score) and +2 payload
    for (int i = lane; i < q_len; i += 32) {
        bvec[i] = i == q_len - 1 ? 0 : kPad;          // rows the sweep does not reach keep these
        bvec[q_len + i] = kPad;
        bvec[2 * q_len + i] = kPad;
    }
    __syncwarp();
    int best = 0;
    for (int s = 0; s < n_stripes; ++s) {
        __syncwarp();
        build_profile2(prof, q, q_len, tk.reverse != 0, true, s * kRows, lane, sc);
        __syncwarp();
        const int4* bin = bnd + (size_t)((s + 1) & 1) * t_len;
        int4* bout = bnd + (size_t)(s & 1) * t_len;
        const bool top = s > 0, bot = s + 1 < n_stripes;
        int H[kR], E1[kR], E2[kR];
#pragma unroll
        for (int r = 0; r < kR; ++r) { H[r] = 0; E1[r] = sc.open1; E2[r] = sc.open2; }
        int hup_prev = 0, h_out = 0, f1_out = 0, f2_out = 0;
        int4 bcur = make_int4(0, 0, 0, 0);
        const int nsteps = t_len + 31;
        // One column step of this lane.  PLAIN: every lane's column lies outside the window and before the last column
        // (off >= 11): no payload, nothing to capture -- the body the sweep runs for all but its last 42 steps.
        auto step = [&](int st, auto plain_tag) {
            constexpr bool PLAIN = decltype(plain_tag)::value;
            if (top && (st & 31) == 0) {
                const int cj = st + lane;
                bcur = cj < t_len ? __ldcg(&bin[cj]) : make_int4(0, 0, 0, 0);
            }
            int hup = __shfl_up_sync(kFull, h_out, 1);
            int f1 = __shfl_up_sync(kFull, f1_out, 1);
            int f2 = __shfl_up_sync(kFull, f2_out, 1);
            if (top) {
                const int bh = __shfl_sync(kFull, bcur.x, st & 31), bf1 = __shfl_sync(kFull, bcur.y, st & 31), bf2 = __shfl_sync(kFull, bcur.z, st & 31);
                if (lane == 0) { hup = bh; f1 = bf1; f2 = bf2; }
            } else if (lane == 0) { hup = 0; f1 = kPad; f2 = kPad; }
            const int p = st - lane;                 // reversed column; it consumes the right anchor's base off = t_len - 1 - p
            if (p >= 0 && p < t_len) {
                const int off = t_len - 1 - p;
                const int code = (tw[p >> 4] >> (30 - 2 * (p & 15))) & 3;
                const bool in_diag = !PLAIN && off < 10;
                const bool in_next = !PLAIN && off - 1 < 10 && off >= 1;       // the next reversed column's base
                const bool in_ins = !PLAIN && off < 9;                         // insertions at right-anchor position off (tk.py:477)
                const int h_open_pay = in_next ? -4 : 0, h_ext_pay = in_next ? (off - 1 == 9 ? -4 : -2) : 0;
                const int v_open_pay = in_ins ? -4 : 0, v_ext_pay = in_ins ? -2 : 0;
                const int ho1 = sc.open1 + h_open_pay, ho2 = sc.open2 + h_open_pay, he1 = sc.ext1 + h_ext_pay, he2 = sc.ext2 + h_ext_pay;
                const int vo1 = sc.open1 + v_open_pay, vo2 = sc.open2 + v_open_pay, ve1 = sc.ext1 + v_ext_pay, ve2 = sc.ext2 + v_ext_pay;
                const int* pr = prof + ((in_diag ? 4 : 0) + code) * kRows + lane * kR;
                const bool last = !PLAIN && p == t_len - 1;
                int hd = hup_prev;
                hup_prev = hup;
                int cm = best;
                if (last) {           // the gap states that ENTER the last column (they consume it): the spanning-gap joins
#pragma unroll
                    for (int r = 0; r < kR; ++r) {
                        const int i = q_len - 2 - (s * kRows + lane * kR + r);
                        if (i >= 0) { bvec[q_len + i] = E1[r] + refund1; bvec[2 * q_len + i] = E2[r] + refund2; }
                    }
                }
#pragma unroll
                for (int r = 0; r < kR; ++r) {
                    const int hleft = H[r];
                    const int t = __vimax3_s32(hd + pr[r], E1[r], E2[r]);
                    const int h = __vimax3_s32_relu(t, f1, f2);
                    E1[r] = __viaddmax_s32(h, ho1, E1[r] + he1);
                    E2[r] = __viaddmax_s32(h, ho2, E2[r] + he2);
                    f1 = __viaddmax_s32(h, vo1, f1 + ve1);
                    f2 = __viaddmax_s32(h, vo2, f2 + ve2);
                    hd = hleft;
                    H[r] = h;
                    if (r & 1) cm = __vimax3_s32(cm, h, H[r - 1]);
                }
                if (last) {
#pragma unroll
                    for (int r = 0; r < kR; ++r) {
                        const int i = q_len - 2 - (s * kRows + lane * kR + r);
                        if (i >= 0) bvec[i] = H[r];
                    }
                }
                best = cm;
                h_out = H[kR - 1]; f1_out = f1; f2_out = f2;
                if (bot && lane == 31) __stcg(&bout[p], make_int4(h_out, f1_out, f2_out, 0));
            }
        };
        int st = 0;
        for (const int plain_end = min(nsteps, t_len - 11); st < plain_end; ++st) step(st, std::true_type{});   // lane 0's off >= 11
        for (; st < nsteps; ++st) step(st, std::false_type{});
        __syncwarp();
        __threadfence_block();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(kFull, best, o));
    if (lane == 0) *ronly = best;
}

// ---- forward sweep of one (read, strand, k1) with a junction per k2 ----------------------------------------------------
template <int MODE>
__device__ __forceinline__ void ladder_fwd_task(const LadFwdTask& tk, const uint32_t* __restrict__ pool, const WinScore& sc,
                                                int* prof, int* bsm, int* jbest, int* pbest, int4* bnd, const int* __restrict__ bvec,
                                                int ronly, int* cstate, int* pbest1, int2* out, int lane) {
    const uint32_t* q = pool + tk.q_word;
    const uint32_t* tw = pool + tk.t_word;
    const int q_len = tk.q_len, a = tk.win_a;
    const int c_first = tk.n_pre + tk.m2 * tk.k2_first, c_step = tk.m2 * tk.k2_step;
    const int t_len = tk.n_pre + tk.m2 * (tk.k2_first + tk.k2_step * (tk.k2_count - 1));
    const int n_stripes = (q_len + kRows - 1) / kRows;
    for (int j = lane; j < tk.k2_count; j += 32) { jbest[j] = 0; pbest[j] = 0; }
    int* cst = cstate + tk.cstate;                     // kPrefix: [k][3][q_len] to fill; kCont: [3][q_len] to start from
    for (int s = 0; s < n_stripes; ++s) {
        int best = 0;                                  // of this stripe's rows, columns up to the lane's current one
        __syncwarp();
        build_profile2(prof, q, q_len, tk.reverse != 0, false, s * kRows, lane, sc);
        if (MODE != kPrefix) {
#pragma unroll
            for (int r = 0; r < kR; ++r) {
                const int i = s * kRows + lane * kR + r;
#pragma unroll
                for (int c = 0; c < 3; ++c) bsm[c * kRows + lane * kR + r] = i < q_len ? __ldcg(&bvec[c * q_len + i]) : kPad;
            }
        }
        __syncwarp();
        const int4* bin = bnd + (size_t)((s + 1) & 1) * t_len;
        int4* bout = bnd + (size_t)(s & 1) * t_len;
        const bool top = s > 0, bot = s + 1 < n_stripes;
        int H[kR], E1[kR], E2[kR];
        int hup_prev = 0, h_out = 0, f1_out = 0, f2_out = 0;
#pragma unroll
        for (int r = 0; r < kR; ++r) { H[r] = 0; E1[r] = sc.open1; E2[r] = sc.open2; }
        if (MODE == kCont) {                           // the column this k1's templates continue from
            const int row0 = s * kRows + lane * kR;
#pragma unroll
            for (int r = 0; r < kR; ++r)
                if (row0 + r < q_len) { H[r] = __ldcg(&cst[row0 + r]); E1[r] = __ldcg(&cst[q_len + row0 + r]); E2[r] = __ldcg(&cst[2 * q_len + row0 + r]); }
            if (row0 >= 1 && row0 - 1 < q_len) hup_prev = __ldcg(&cst[row0 - 1]);
        }
        int4 bcur = make_int4(0, 0, 0, 0);
        int jidx = 0, jcol = c_first;                  // the next junction of this lane: grid point jidx after jcol columns (>= 1)
        const int nsteps = t_len + 31;
        // One column step of this lane.  PLAIN: every lane's column lies before the window (p + 1 < a, so before every
        // junction too): no payload, nothing to join or save -- the body of most of a sweep over a long left anchor.
        auto step = [&](int st, auto plain_tag) {
            constexpr bool PLAIN = decltype(plain_tag)::value;
            if (top && (st & 31) == 0) {
                const int cj = st + lane;
                bcur = cj < t_len ? __ldcg(&bin[cj]) : make_int4(0, 0, 0, 0);
            }
            int hup = __shfl_up_sync(kFull, h_out, 1);
            int f1 = __shfl_up_sync(kFull, f1_out, 1);
            int f2 = __shfl_up_sync(kFull, f2_out, 1);
            if (top) {
                const int bh = __shfl_sync(kFull, bcur.x, st & 31), bf1 = __shfl_sync(kFull, bcur.y, st & 31), bf2 = __shfl_sync(kFull, bcur.z, st & 31);
                if (lane == 0) { hup = bh; f1 = bf1; f2 = bf2; }
            } else if (lane == 0) { hup = 0; f1 = kPad; f2 = kPad; }
            const int p = st - lane;
            if (p >= 0 && p < t_len) {
                const int code = (tw[p >> 4] >> (30 - 2 * (p & 15))) & 3;
                const bool in_diag = !PLAIN && (MODE == kCont || p >= a);     // (every grid point's window reaches past the junction)
                const bool in_next = !PLAIN && (MODE == kCont || p + 1 >= a);
                const bool in_ins = !PLAIN && (MODE == kCont || p + 1 > a);
                const int h_open_pay = in_next ? -4 : 0, h_ext_pay = in_next ? (MODE != kCont && p + 1 == a ? -4 : -2) : 0;
                const int v_open_pay = in_ins ? -4 : 0, v_ext_pay = in_ins ? -2 : 0;
                const int ho1 = sc.open1 + h_open_pay, ho2 = sc.open2 + h_open_pay, he1 = sc.ext1 + h_ext_pay, he2 = sc.ext2 + h_ext_pay;
                const int vo1 = sc.open1 + v_open_pay, vo2 = sc.open2 + v_open_pay, ve1 = sc.ext1 + v_ext_pay, ve2 = sc.ext2 + v_ext_pay;
                const int* pr = prof + ((in_diag ? 4 : 0) + code) * kRows + lane * kR;
                const bool junc = !PLAIN && jidx < tk.k2_count && p + 1 == jcol;
                int hd = hup_prev;
                hup_prev = hup;
                int cm = best, jmax = 0;
#pragma unroll
                for (int r = 0; r < kR; ++r) {
                    const int hleft = H[r];
                    const int e1pre = E1[r], e2pre = E2[r];
                    const int t = __vimax3_s32(hd + pr[r], E1[r], E2[r]);
                    const int h = __vimax3_s32_relu(t, f1, f2);
                    E1[r] = __viaddmax_s32(h, ho1, E1[r] + he1);
                    E2[r] = __viaddmax_s32(h, ho2, E2[r] + he2);
                    f1 = __viaddmax_s32(h, vo1, f1 + ve1);
                    f2 = __viaddmax_s32(h, vo2, f2 + ve2);
                    hd = hleft;
                    H[r] = h;
                    if (r & 1) cm = __vimax3_s32(cm, h, H[r - 1]);
                    if (!PLAIN && MODE != kPrefix && junc) {
                        const int x = lane * kR + r;
                        jmax = __vimax3_s32(jmax, h + bsm[x], e1pre + bsm[kRows + x]);
                        jmax = max(jmax, e2pre + bsm[2 * kRows + x]);
                    }
                }
                best = cm;
                if (junc) {
                    if (MODE == kPrefix) {             // the states every template of this k1 continues from
                        const int row0 = s * kRows + lane * kR;
                        int* dst = cst + (size_t)jidx * 3 * q_len;
#pragma unroll
                        for (int r = 0; r < kR; ++r)
                            if (row0 + r < q_len) { __stcg(&dst[row0 + r], H[r]); __stcg(&dst[q_len + row0 + r], E1[r]); __stcg(&dst[2 * q_len + row0 + r], E2[r]); }
                    } else {
                        atomicMax(&jbest[jidx], jmax);
                    }
                    atomicMax(&pbest[jidx], best);
                    ++jidx;
                    jcol += c_step;
                }
                h_out = H[kR - 1]; f1_out = f1; f2_out = f2;
                if (bot && lane == 31) __stcg(&bout[p], make_int4(h_out, f1_out, f2_out, 0));
            }
        };
        int st = 0;
        if (MODE != kCont)
            for (const int plain_end = min(nsteps, a - 1); st < plain_end; ++st) step(st, std::true_type{});   // lane 0: p + 1 < a
        for (; st < nsteps; ++st) step(st, std::false_type{});
        __syncwarp();
        __threadfence_block();
    }
    __syncwarp();
    if (MODE == kPrefix) {
        for (int j = lane; j < tk.k2_count; j += 32) pbest1[tk.out_off + j] = pbest[j];
        __threadfence();
    } else {
        const int before = MODE == kCont ? max(ronly, __ldcg(&pbest1[tk.pbest1])) : ronly;
        for (int j = lane; j < tk.k2_count; j += 32) {
            const int w = max(max(pbest[j], jbest[j]), before);
            const int score = (w + 0x8000) >> 16;
            out[tk.out_off + j] = make_int2(score, w - (score << 16));
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(32 * kWarps)
ladder_bwd_kernel(const LadBwdTask* __restrict__ tasks, int n_tasks, const uint32_t* __restrict__ pool, WinScore sc, int4* scratch,
                  int scratch_stride, int* counter, int* bvec, int* ronly) {
    extern __shared__ int wsmem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int* prof = wsmem + warp * (8 * kRows);
    int4* bnd = scratch + (size_t)(blockIdx.x * kWarps + warp) * scratch_stride;
    for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(counter, 1);
        i = __shfl_sync(kFull, i, 0);
        if (i >= n_tasks) break;
        const LadBwdTask tk = tasks[i];
        ladder_bwd_task(tk, pool, sc, prof, bnd, bvec + tk.bvec_off(), ronly + i, lane);
    }
}

__global__ void __launch_bounds__(32 * kWarps)
ladder_fwd_kernel(const LadFwdTask* __restrict__ tasks, int n_tasks, const LadBwdTask* __restrict__ btasks,
                  const uint32_t* __restrict__ pool, WinScore sc, int4* scratch, int scratch_stride, int* counter,
                  const int* __restrict__ bvec, const int* __restrict__ ronly, int* cstate, int* pbest1, int2* out) {
    extern __shared__ int wsmem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int* base = wsmem + warp * (8 * kRows + 3 * kRows + 2 * kMaxK2);
    int* prof = base;
    int* bsm = base + 8 * kRows;
    int* jbest = bsm + 3 * kRows;
    int* pbest = jbest + kMaxK2;
    int4* bnd = scratch + (size_t)(blockIdx.x * kWarps + warp) * scratch_stride;
    for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(counter, 1);
        i = __shfl_sync(kFull, i, 0);
        if (i >= n_tasks) break;
        const LadFwdTask tk = tasks[i];
        if (tk.mode == kPrefix)
            ladder_fwd_task<kPrefix>(tk, pool, sc, prof, bsm, jbest, pbest, bnd, bvec, 0, cstate, pbest1, out, lane);
        else if (tk.mode == kCont)
            ladder_fwd_task<kCont>(tk, pool, sc, prof, bsm, jbest, pbest, bnd, bvec + btasks[tk.bwd].bvec_off(), ronly[tk.bwd], cstate, pbest1, out, lane);
        else
            ladder_fwd_task<kWhole>(tk, pool, sc, prof, bsm, jbest, pbest, bnd, bvec + btasks[tk.bwd].bvec_off(), ronly[tk.bwd], cstate, pbest1, out, lane);
    }
}

}  // namespace nrw
