// nr_pair_kernels.cuh -- paired DP kernels: TWO reads per warp, one per 16-bit half of every DP word (u16x2).
//
// Same contract as nr_kernels.cuh (oracle/nr_oracle.c), same wavefront mapping (one warp per task, lane l owns R rows,
// skewed column sweep, query profile in shared memory); what changes is the DP word.  Rounds 2 and 3 of the reference
// (nanoRepeat_bam.py:349-384, :408-434, :452-500) read, per alignment, the score, tend (round 2) and two span
// predicates -- never a coordinate that needs 16 bits of its own -- so a cell fits 16 bits and a DPX instruction
// (VIADDMNMX.U16x2 / VIMNMX3.U16x2) updates one cell of each of two reads of the same region (same template):
//
//     w = 2 * score + u + 64        u = 1: the alignment did NOT start in the marked prefix of the template
//                                          (round 2: columns <= |left|, :373; round 3: columns < |left|, :427)
//
// * unsigned halves with a bias of 64: no half ever goes below 0 (the deepest value is floor - open2 - ext2 = 13), so a
//   plain 32-bit add of a two-half constant cannot borrow across the halves and the five adds of the cell stay IMADs
//   on the FMA pipe, beside the DPX pipe;
// * a fresh start is the word 65 (score 0, unmarked); it enters as the third operand of the diagonal's VIADDMNMX, so the
//   cell is 7 DPX-class instructions + 4 IMAD per PAIR of cells (3.5 DPX per cell against 6 for the 32-bit word);
// * when a lane has finished the last marked column, every live state with a positive score loses 1 (becomes "started
//   inside"); integer max then prefers the unmarked word among equal scores, which is the contract's "largest tstart".
//
// Round 3 (pair_ladder_kernel) shares prefix and suffix over the rungs exactly like ladder_kernel: one backward sweep
// over reverse(right), one forward sweep over left + motif^kmax, junction candidates forward + backward at every column
// |left| + k * |motif|.  The backward words carry the score only, so among candidates of equal total the contract's
// order (smallest tend, then largest tstart) is not decidable when a marked and an unmarked candidate tie for a rung
// that ties for the read's top score: those reads (none in the five configs' synthetic data, a few in the crafted
// tests) are appended to a redo list and rescored by the 32-bit flag ladder right behind this kernel.  Everything
// else -- scores, the "ends in right" predicate, the selection -- is exact as computed here.
#pragma once
#include "nr_kernels.cuh"

namespace nr {
namespace pr {

typedef unsigned u32;
constexpr int kBias = 64;
__host__ __device__ constexpr u32 pk2(int hi, int lo) { return ((u32)(hi & 0xffff) << 16) | (u32)(lo & 0xffff); }
__host__ __device__ constexpr u32 pk(int v) { return pk2(v, v); }
// 32-bit addend that subtracts v from both halves (valid while both halves stay >= v)
__host__ __device__ constexpr u32 sub2(int v) { return 0u - (((u32)v << 16) | (u32)v); }

// map-ont (the reference's only scoring, tk.py:502-517) in doubled units: bit 0 of a word is the mark
constexpr int kMatch = 4, kMismatch = 8, kAmbiguous = 2, kOpen1 = 12, kExt1 = 4, kOpen2 = 50, kExt2 = 2, kRefund1 = 8, kRefund2 = 48;
constexpr u32 kFloorFwd = pk(kBias + 1);     // score 0, unmarked
constexpr u32 kFloorBwd = pk(kBias);         // backward words: bit 0 stays clear, so forward + backward keeps the mark
constexpr u32 kOnes = 0x00010001u;

__device__ __forceinline__ u32 pmadd(u32 a, u32 mul, u32 b) {
    u32 d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(mul), "r"(b));
    return d;
}

// One cell of both reads.  hd: H(i-1, j-1); s: substitution increment per half (two's complement halves).
template <u32 FLOOR>
__device__ __forceinline__ void cell(u32 hd, u32 s, u32 one, u32& h, u32& e1, u32& e2, u32& f1, u32& f2) {
    const u32 d = __viaddmax_u16x2(hd, s, FLOOR);
    const u32 t = __vimax3_u16x2(d, e1, e2);
    h = __vimax3_u16x2(t, f1, f2);
    e1 = __viaddmax_u16x2(h, pk(-kOpen1), pmadd(e1, one, sub2(kExt1)));
    e2 = __viaddmax_u16x2(h, pk(-kOpen2), pmadd(e2, one, sub2(kExt2)));
    f1 = __viaddmax_u16x2(h, pk(-kOpen1), pmadd(f1, one, sub2(kExt1)));
    f2 = __viaddmax_u16x2(h, pk(-kOpen2), pmadd(f2, one, sub2(kExt2)));
}

struct Pair2 {         // round 2: two tasks of one region (same template); b < 0: no partner
    int32_t a, b;
    int32_t mark_col;  // |left|: an alignment that starts at a column <= mark_col passes the span test (:373)
    int32_t state_off; // where the pair's DP state after column |left| - 2 is kept for round 3 (units of 32 words), -1: not kept
    int32_t check_col; // single-stripe pairs: first column of the dominance exit's checks (Sweep::run); -1: no exit
    int32_t period;    // lcm(16, |motif|): columns between two checks
    int32_t pad[2];
};

// d_counters slots of a round-2 launch: cells the dominance exit skipped, per half (rows x columns, padding included),
// and (rows of real reads) x columns x 32, both as 64-bit sums
constexpr int kExitSlot = 24;

struct Pair3 {         // round 3: two LadderTasks of one region, either may be absent (< 0)
    int32_t a, b;
    int32_t rung_off;  // first (P, J) token pair of this pair in the rung buffer
    int32_t state_off; // >= 0: the forward sweep resumes from the state round 2 kept (same pair, same halves, same R)
    int32_t R;         // rows per lane (the pair's shape in round 2 when it resumes; 0: from the reads' lengths)
    int32_t pad[3];
};

// words per lane of a kept state: H, E1, E2 of R rows and the lane's best prefix class
__host__ __device__ constexpr int state_words(int R) { return 3 * R + 1; }

// Query profile of a pair: prof[(c * CH + chunk) * 32 + lane].{x,y,z,w} = increments of rows 4*chunk..+3 of this lane
// against target code c, read A in the high half, read B in the low half.  Rows past a read's end score as mismatches:
// they lie below every real row, nothing flows upwards, and whatever they hold is below a real cell of the same or an
// earlier column, so they can neither set nor tie a maximum.
template <int R>
__device__ __forceinline__ void build_profile(uint4* prof, const uint32_t* __restrict__ qa, int q_a,
                                              const uint32_t* __restrict__ qb, int q_b, int row0, int lane, bool reverse) {
    constexpr int CH = StripeCfg<R>::CH;
    u32* p = reinterpret_cast<u32*>(prof);
    // a read base other than ACGT (code 5) scores -sc_ambi against every template base (nr_kernels.cuh, build_profile)
    const uint32_t amb_a = q_a > 0 ? read_ambiguity_plane(qa, q_a) : 0u, amb_b = q_b > 0 ? read_ambiguity_plane(qb, q_b) : 0u;
#pragma unroll
    for (int r = 0; r < 4 * CH; ++r) {
        const int i = row0 + r;
        int ca = 4, cb = 4;
        if (r < R && i < q_a) {
            const int qi = reverse ? q_a - 1 - i : i;
            ca = (qa[qi >> 4] >> (30 - 2 * (qi & 15))) & 3;
            if (amb_a && read_base_ambiguous(qa, amb_a, qi)) ca = 5;
        }
        if (r < R && i < q_b) {
            const int qi = reverse ? q_b - 1 - i : i;
            cb = (qb[qi >> 4] >> (30 - 2 * (qi & 15))) & 3;
            if (amb_b && read_base_ambiguous(qb, amb_b, qi)) cb = 5;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
            p[((c * CH + (r >> 2)) * 32 + lane) * 4 + (r & 3)] =
                pk2(ca == 5 ? -kAmbiguous : ca == c ? kMatch : -kMismatch, cb == 5 ? -kAmbiguous : cb == c ? kMatch : -kMismatch);
    }
}

constexpr int kP2 = 0, kPB = 1, kPF = 2;

// One sweep of one pair (single stripe).
//   kP2: round 2, read x left + motif^T; marks after column mark_col; per half the first column that reaches the
//        best score (tend) and the mark of the best word there.
//   kPB: reversed reads x reverse(right), score only; running maximum (the R-only class); the final column's junction
//        state (H, E1 + refund1, E2 + refund2) goes to bvec in the forward layout, each half at its own read's rows.
//   kPF: reads x left + motif^kmax; marks after column |left| - 1; junction candidates and (P, J) tokens as in
//        nr_kernels.cuh; the last lane stores every rung's token pair.
// MULTI: one stripe of a pair of LONG reads (more than 512 bases): the stripes of the pair run on different warps at the
// same time and hand their bottom rows down through tagged boundary entries exactly like the 32-bit stripes of
// nr_kernels.cuh (load_bnd / store_bnd: a boundary entry holds H, F1, F2 as three 32-bit words -- here each is the two
// halves of the pair).  `top`: a stripe above exists (lane 0 takes its upper neighbour from bnd_in); `bot`: one below.
template <int R, int MODE, bool MULTI = false>
struct Sweep {
    static constexpr u32 FLOOR = MODE == kPB ? kFloorBwd : kFloorFwd;
    static constexpr bool kMarks = MODE != kPB;
    // inputs
    bool top, bot;
    const ulonglong2* bnd_in;
    ulonglong2* bnd_out;
    int tag_in, tag_out;
    int* spin;
    int4 bcur;
    ulonglong2 bnxt;
    // MULTI, forward sweep of a long pair: the junction vectors come from the backward stripes (global `bstage`,
    // [state][reversed row] of two-half words) once all of them are done; tokens travel between the stripes as tagged
    // 16-byte entries like those of nr_kernels.cuh
    const ulonglong2* tok_in;
    ulonglong2* tok_out;
    const u32* bstage;
    int b_stride, brow0;           // words per state plane; first forward row of this stripe's lane 0
    const int* bdone;
    int bdone_need;
    bool late_pending;
    u32* bsm_w;
    const uint4* prof;
    const uint32_t* twords;
    int t_len, lane;
    int mark_col;
    int q_a, q_b;
    const u32* bsm;                // kPF: junction vectors, three planes [state][row][lane] of two-half words
    uint2* rung_out;
    int jnext, m, kcnt, zone_start; // zone_start: in steps of this sweep
    int col0;                      // first column of the sweep (kPF resuming from a kept state: |left| - 1; else 0)
    const u32* resume;             // kPF: state kept by round 2, [word * 32 + lane]
    u32* save;                     // kP2: where to keep the state after column save_col (null: nowhere)
    int save_col;
    bool exits;                    // kP2 dominance exit: on for this pair (the kept cut follows the profile in shared memory)
    int check_col, period;
    int next_check;                // step of the next check (-1: none)
    int exit_st;                   // step at which the exit ended the sweep (-1: swept to the end)
    u32* kept_io;                  // global, this warp's slot: the kept cut's hup_prev, f1_out, f2_out and the period,
                                   // [word * 32 + lane] (no room in registers or in shared memory at R = 16)
    // state
    u32 H[R], E1[R], E2[R];
    u32 hup_prev, h_out, f1_out, f2_out;
    u32 best;                      // kPB / kPF: running maximum word per half
    u32 bestc, raw_hi, raw_lo;     // kP2: best score class per half ((word | 1)); the best word itself (its mark)
    int st_hi, st_lo;              // kP2: step at which each half's class was first reached
    u32 nz, bz;                    // lane 0: what SHFL.UP "delivers" is replaced by the matrix border (x * nz + bz)
    uint32_t twl, w0, w1;
    int wi, wmax, wsh;
    const char* prof_lane;
    u32 tokP, tokJ;

    __device__ __forceinline__ uint32_t tword(int i) const { return __ldg(&twords[min(max(i, 0), wmax)]); }

    __device__ __forceinline__ void init() {
        if (MODE == kPF && resume) {
            // round 2 swept these reads over the same left anchor with the same pairing: take over where every live
            // state is still unmarked in both rounds (after column |left| - 2)
#pragma unroll
            for (int r = 0; r < R; ++r) {
                H[r] = __ldcg(&resume[r * 32 + lane]);
                E1[r] = __ldcg(&resume[(R + r) * 32 + lane]);
                E2[r] = __ldcg(&resume[(2 * R + r) * 32 + lane]);
            }
            hup_prev = lane ? __ldcg(&resume[(R - 1) * 32 + lane - 1]) : FLOOR;
            best = __ldcg(&resume[3 * R * 32 + lane]);
        } else {
#pragma unroll
            for (int r = 0; r < R; ++r) { H[r] = FLOOR; E1[r] = FLOOR + sub2(kOpen1); E2[r] = FLOOR + sub2(kOpen2); }
            hup_prev = FLOOR;
            best = 0;
        }
        h_out = FLOOR; f1_out = FLOOR; f2_out = FLOOR;
        bestc = FLOOR | kOnes; raw_hi = 0; raw_lo = 0; st_hi = 0; st_lo = 0;
        nz = lane != 0; bz = lane != 0 ? 0u : FLOOR;
        wmax = (t_len + 15) >> 4;
        wi = (col0 - lane) >> 4;
        wsh = 2 * ((col0 - lane) & 15);
        w0 = tword(wi); w1 = tword(wi + 1);
        twl = 0;
        prof_lane = reinterpret_cast<const char*>(prof + lane);
        tokP = 0; tokJ = 0;
        if (MULTI) {
            bcur = make_int4(0, 0, 0, 0); bnxt = make_ulonglong2(0ull, 0ull);
            if (top) bnxt = load_bnd(&bnd_in[lane < t_len ? lane : t_len - 1]);      // validated when it is taken over
            late_pending = MODE == kPF;
        }
    }

    __device__ __forceinline__ void refill() {
        twl = __funnelshift_l(w1, w0, wsh);
        w0 = w1;
        ++wi;
        w1 = tword(wi + 1);
    }

    __device__ __forceinline__ unsigned next_base(unsigned four) {
        unsigned lo, hi;
        asm("{\n\t.reg .u64 p;\n\tmul.wide.u32 p, %2, %3;\n\tmov.b64 {%0, %1}, p;\n\t}" : "=r"(lo), "=r"(hi) : "r"(twl), "r"(four));
        twl = lo;
        return hi;
    }

    // JUNC: junction candidates of this column (forward word + backward word per row and state; the sums are plain 32-bit
    // adds -- both halves stay below 2^16 -- on the FMA pipe, the maxima three-input ones: 1.5 DPX-class instructions
    // per row instead of 3).  KEEP_E (kPB, guarded steps): in the sweep's last column the gap states are left as they
    // entered it, which is what the junction vectors hold (store_junction_vectors).
    template <bool JUNC, bool KEEP_E = false>
    __device__ __forceinline__ u32 cells(const uint4* pp, u32 hd, u32 cm, u32& f1, u32& f2, u32 one, u32& jhi, bool keep = false) {
        constexpr int CH = StripeCfg<R>::CH;
        u32 jprev = 0;
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const uint4 sv = pp[c * 32];
            const u32 s4[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int r = 4 * c + u;
                if (r < R) {
                    const u32 hleft = H[r];
                    const u32 e1pre = E1[r], e2pre = E2[r];
                    u32 h;
                    cell<FLOOR>(hd, s4[u], one, h, E1[r], E2[r], f1, f2);
                    if (KEEP_E) { E1[r] = keep ? e1pre : E1[r]; E2[r] = keep ? e2pre : E2[r]; }
                    if (JUNC) {
                        const u32 bx = bsm[(0 * R + r) * 32 + lane], by = bsm[(1 * R + r) * 32 + lane], bz = bsm[(2 * R + r) * 32 + lane];
                        const u32 t = __vimax3_u16x2(pmadd(h, one, bx), pmadd(e1pre, one, by), pmadd(e2pre, one, bz));
                        if (r & 1) jhi = __vimax3_u16x2(jhi, jprev, t);
                        else if (r == R - 1) jhi = __vmaxu2(jhi, t);
                        jprev = t;
                    }
                    hd = hleft;
                    H[r] = h;
                    if (r & 1) cm = __vimax3_u16x2(cm, h, H[r - 1]);
                    else if (r == R - 1) cm = __vmaxu2(cm, h);
                }
            }
        }
        return cm;
    }

    // once per lane, after the last marked column: every live state with a positive score started inside
    __device__ __forceinline__ void mark_started_inside() {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            H[r] = __viaddmax_u16x2(H[r], pk(-1), FLOOR);
            E1[r] = __viaddmax_u16x2(E1[r], pk(-1), __vminu2(E1[r], FLOOR));
            E2[r] = __viaddmax_u16x2(E2[r], pk(-1), __vminu2(E2[r], FLOOR));
        }
        hup_prev = __viaddmax_u16x2(hup_prev, pk(-1), FLOOR);
    }

    // MULTI forward sweep: fetch this stripe's junction vectors when the sweep reaches its first junction column, so that
    // the forward stripes run beside the backward ones.  Forward row i of read A is reversed row q_a - 2 - i (B: q_b - 2 - i).
    __device__ __forceinline__ void late_load() {
        wait_cols(bdone, bdone_need, lane, spin);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int idx0 = brow0 + lane * R + r;
            const int ia = q_a - 2 - idx0, ib = q_b - 2 - idx0;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const u32 da = c == 0 ? (idx0 < q_a ? (u32)kBias : 0u) : 0u, db = c == 0 ? (idx0 < q_b ? (u32)kBias : 0u) : 0u;
                const u32 a = ia >= 0 ? __ldcg(&bstage[c * b_stride + ia]) >> 16 : da;
                const u32 b = ib >= 0 ? __ldcg(&bstage[c * b_stride + ib]) & 0xffffu : db;
                bsm_w[(c * R + r) * 32 + lane] = (a << 16) | b;
            }
        }
        __syncwarp();
        late_pending = false;
    }

    // MULTI backward sweep, after the stripe: H of the last column and the gap states that entered it, by reversed row
    __device__ __forceinline__ void store_stage(u32* stage, int stride, int row0) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = row0 + lane * R + r;
            __stcg(&stage[0 * stride + i], H[r]);
            __stcg(&stage[1 * stride + i], E1[r] + pk(kRefund1));
            __stcg(&stage[2 * stride + i], E2[r] + pk(kRefund2));
        }
    }

    // kPB, after the sweep: the junction vectors.  Every lane still holds, for its R rows of the reversed reads, H of the
    // last column and the gap states that entered it (cells<.., KEEP_E>).  They go to `stage` (the reversed profile's
    // shared memory, dead by now) as they are, [state][row][lane]; then every lane gathers the vectors of ITS forward
    // rows -- forward row i of read A is reversed row q_a - 2 - i (read B: q_b - 2 - i; the halves move apart) -- and
    // writes them in the forward layout the junction columns read.  Rows the sweep has no value for: the right part is
    // empty (score 0, no gap state) for the last row of a read, void below it.
    __device__ __forceinline__ void store_junction_vectors(u32* stage, u32* bvec_fwd) {
        __syncwarp();
#pragma unroll
        for (int r = 0; r < R; ++r) {
            stage[(0 * R + r) * 32 + lane] = H[r];
            stage[(1 * R + r) * 32 + lane] = E1[r] + pk(kRefund1);
            stage[(2 * R + r) * 32 + lane] = E2[r] + pk(kRefund2);
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int idx0 = lane * R + r;
            const int ia = q_a - 2 - idx0, ib = q_b - 2 - idx0;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const u32 da = c == 0 ? (idx0 < q_a ? (u32)kBias : 0u) : 0u, db = c == 0 ? (idx0 < q_b ? (u32)kBias : 0u) : 0u;
                const u32 a = ia >= 0 ? stage[(c * R + ia % R) * 32 + ia / R] >> 16 : da;
                const u32 b = ib >= 0 ? stage[(c * R + ib % R) * 32 + ib / R] & 0xffffu : db;
                bvec_fwd[(c * R + r) * 32 + lane] = (a << 16) | b;
            }
        }
    }

    // TRACK (kP2): per half the step of the last strict improvement of the score class; without it (the columns an
    // alignment that passes the span test cannot end in) only the running maximum word.
    // FAST: every lane is inside the matrix, no bounds checks.  SPECIAL (with FAST): the step may still hold a lane at a
    // junction, at the last marked column or at the column whose state is kept -- the guard-free body with those checks.
    template <bool FAST, bool TRACK, bool SPECIAL = false>
    __device__ __forceinline__ void step(int st, u32 one, unsigned four) {
        const bool zone = MODE == kPF && (FAST ? SPECIAL : st >= zone_start);     // uniform
        constexpr int CH = StripeCfg<R>::CH;
        u32 hup = __shfl_up_sync(kFull, h_out, 1);
        u32 f1 = __shfl_up_sync(kFull, f1_out, 1);
        u32 f2 = __shfl_up_sync(kFull, f2_out, 1);
        u32 tP = 0, tJ = 0;
        if (zone) {
            tP = __shfl_up_sync(kFull, tokP, 1);
            tJ = __shfl_up_sync(kFull, tokJ, 1);
        }
        if (MULTI && top) {                 // uniform branch: lane 0's upper neighbour is the stripe above
            if ((st & 31) == 0) {
                ulonglong2 raw = bnxt;
                const int cj = st + lane;
                for (int tries = 0; !__all_sync(kFull, bnd_valid(raw, tag_in) || cj >= t_len); ++tries) {
                    if (tries > kSpinLimit) { *spin = 1; break; }
                    if (tries > 3) __nanosleep(32);
                    raw = load_bnd(&bnd_in[cj < t_len ? cj : t_len - 1]);
                }
                bcur = unpack_bnd(raw);
                const int nj = st + 32 + lane;
                bnxt = load_bnd(&bnd_in[nj < t_len ? nj : t_len - 1]);      // in flight for the next 32 steps
            }
            const u32 bh = __shfl_sync(kFull, (u32)bcur.x, st & 31);
            const u32 bf1 = __shfl_sync(kFull, (u32)bcur.y, st & 31);
            const u32 bf2 = __shfl_sync(kFull, (u32)bcur.z, st & 31);
            if (lane == 0) { hup = bh; f1 = bf1; f2 = bf2; }
        } else {
            hup = pmadd(hup, nz, bz);
            f1 = pmadd(f1, nz, bz);
            f2 = pmadd(f2, nz, bz);
        }
        const unsigned tb = next_base(four);
        const int rel = st - lane;
        const int jj = rel + col0;
        const bool anyj = zone && __any_sync(kFull, jj + 1 == jnext && jj < t_len);
        if (FAST || (rel >= 0 && jj < t_len)) {
            const uint4* pp = reinterpret_cast<const uint4*>(prof_lane + tb * (unsigned)(CH * 512));
            const u32 hd = hup_prev;
            hup_prev = hup;
            constexpr bool kChecks = !FAST || SPECIAL;
            const bool last_col = !FAST && MODE == kPB && jj == t_len - 1;
            u32 cm, jhi = 0;
            const u32 cm0 = (MODE == kP2 && TRACK) ? 0u : best;
            if (zone && anyj) cm = cells<true>(pp, hd, cm0, f1, f2, one, jhi);
            else if (MODE == kPB && !FAST) cm = cells<false, true>(pp, hd, cm0, f1, f2, one, jhi, last_col);
            else cm = cells<false>(pp, hd, cm0, f1, f2, one, jhi);
            h_out = H[R - 1]; f1_out = f1; f2_out = f2;
            if (MODE == kP2 && TRACK) {
                // per half: a strictly higher score class (the mark bit forced on both sides); the first column wins
                // (not __vibmax_u16x2: its inline asm re-reads an input after writing its output without an early clobber,
                // so "best = __vibmax(best, ...)" may alias the two and report "kept" for ever)
                const u32 nb = __vmaxu2(bestc, cm | kOnes);
                const u32 x = nb ^ bestc;
                bestc = nb;
                if (x > 0xffffu) { st_hi = st; raw_hi = cm; }
                if (x & 0xffffu) { st_lo = st; raw_lo = cm; }
                if (kChecks && save && jj == save_col) {    // the state round 3 resumes from
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        __stcg(&save[r * 32 + lane], H[r]);
                        __stcg(&save[(R + r) * 32 + lane], E1[r]);
                        __stcg(&save[(2 * R + r) * 32 + lane], E2[r]);
                    }
                    __stcg(&save[3 * R * 32 + lane], bestc);
                }
            } else {
                best = cm;
            }
            if (zone && jj + 1 == jnext) {
                if (lane == 0) {
                    tP = 0; tJ = 0;
                    if (MULTI && top) {     // both 64-bit elements of the token carry the tag in their upper half
                        ulonglong2 t = load_tok(&tok_in[kcnt]);
                        for (int tries = 0; (int)(t.x >> 32) != tag_in || (int)(t.y >> 32) != tag_in; ++tries) {
                            if (tries > kSpinLimit) { *spin = 1; break; }
                            if (tries > 3) __nanosleep(32);
                            t = load_tok(&tok_in[kcnt]);
                        }
                        tP = (u32)t.x; tJ = (u32)t.y;
                    }
                }
                // rung 0's junction column is the last marked column: every forward part that scores started inside
                // but is marked only after this step (candidates with an empty forward part are the R-only class again)
                const u32 jv = jj == mark_col ? jhi - kOnes : jhi;
                tokP = __vmaxu2(tP, best);
                tokJ = __vmaxu2(tJ, jv);
                if (lane == 31) {
                    if (MULTI && bot) __stcg(&tok_out[kcnt], make_ulonglong2(tokP | ((u64)(unsigned)tag_out << 32), tokJ | ((u64)(unsigned)tag_out << 32)));
                    else rung_out[kcnt] = make_uint2(tokP, tokJ);
                }
                jnext += m;
                ++kcnt;
            }
            if (kMarks && kChecks && jj == mark_col) mark_started_inside();
            if (MULTI && bot && lane == 31) store_bnd(&bnd_out[jj], (int)h_out, (int)f1_out, (int)f2_out, tag_out);
        }
    }

    __device__ __forceinline__ void slow_until(int& st, int end, u32 one, unsigned four) {
#pragma unroll 1
        for (; st < end; ++st) {
            if (MULTI && MODE == kPF && late_pending && st >= zone_start) late_load();
            if ((st & 15) == 0) refill();
            step<false, true>(st, one, four);
        }
    }

    // steps per trip of the guard-free loop.  Round 3's warps are spread over several loop variants (backward sweep,
    // forward sweep in and out of the junction zone; for long pairs three per stripe) and the kernel is sensitive to
    // instruction fetch: with four steps per trip (11 KB of code per variant) config 2's launch took anywhere between
    // 1.26 and 1.41 ms from build to build of the library (same kernel code, another place in memory), with two
    // 1.24-1.25 ms on every build and box tried, with one 1.23-1.27 ms.  So: two for single-stripe pairs, one for the
    // stripes of long pairs; round 2 has one loop variant per launch and is fastest with four (1.23 against 1.25 ms).
#ifndef NR_PAIR3_UNROLL
#define NR_PAIR3_UNROLL 2
#endif
#ifndef NR_PAIR2_UNROLL
#define NR_PAIR2_UNROLL 4
#endif
#ifndef NR_PAIR2_MULTI_UNROLL
#define NR_PAIR2_MULTI_UNROLL 4
#endif
    static constexpr int kUnroll = MODE == kP2 ? (MULTI ? NR_PAIR2_MULTI_UNROLL : NR_PAIR2_UNROLL) : (MULTI ? 1 : NR_PAIR3_UNROLL);
    // EXIT (kP2 single stripes): the dominance exit's checks at trip boundaries, where every lane is at the same step
    template <bool TRACK, bool SPECIAL = false, bool EXIT = false>
    __device__ __forceinline__ void fast_until(int& st, int end, u32 one, unsigned four) {
        for (; st + 16 <= end; st += 16) {       // st is a multiple of 16 here
            if (EXIT && st == next_check) {
                if (dominated_then_keep()) { exit_st = st; return; }
                next_check += (int)__ldcg(kept_io + 96 + lane);
            }
            refill();
#pragma unroll 1
            for (int b = 0; b < 16; b += kUnroll) {
#pragma unroll
                for (int u = 0; u < kUnroll; ++u) step<true, TRACK, SPECIAL>(st + b + u, one, four);
            }
        }
    }

    // kP2 dominance exit.  The cut between two steps is everything the rest of the sweep reads: H, E1, E2 of every
    // lane's rows and what is in flight between the lanes (the diagonal hup_prev; h_out is H[R - 1]; f1_out, f2_out).
    // Returns whether the cut is <= the kept one in every half of every word, then keeps the cut.  The 3R planes go
    // behind the profile in shared memory (14 KB per warp at R = 16), the three in-flight words to kept_io.  The first
    // check compares with zeros and fails: no half of a live word is ever 0 (the floor keeps them >= 13).
    __device__ __forceinline__ bool dominated_then_keep() {
        u32* g = kept_io + lane;
        const u32 khp = __ldcg(g), kf1 = __ldcg(g + 32), kf2 = __ldcg(g + 64);
        u32 acc = (__vmaxu2(hup_prev, khp) ^ khp) | (__vmaxu2(f1_out, kf1) ^ kf1) | (__vmaxu2(f2_out, kf2) ^ kf2);
        __stcg(g, hup_prev); __stcg(g + 32, f1_out); __stcg(g + 64, f2_out);
        u32* snap = reinterpret_cast<u32*>(const_cast<uint4*>(prof) + StripeCfg<R>::PROF_INT4);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            u32* k = snap + r * 32 + lane;
            const u32 kh = k[0], ke1 = k[R * 32], ke2 = k[2 * R * 32];
            acc |= (__vmaxu2(H[r], kh) ^ kh) | (__vmaxu2(E1[r], ke1) ^ ke1) | (__vmaxu2(E2[r], ke2) ^ ke2);
            k[0] = H[r]; k[R * 32] = E1[r]; k[2 * R * 32] = E2[r];
        }
        return __all_sync(kFull, acc == 0);
    }

    // zone_start_: kPF, first step (of this sweep) at which a lane can be at a junction column
    __device__ __forceinline__ void run(u32 one, unsigned four, int zone_start_) {
        init();
        zone_start = zone_start_;
        exit_st = -1;
        const int n = t_len - col0;              // columns swept
        const int nsteps = n + 31;
        const int inside_end = ((n - 1) >> 4) << 4;     // steps 31 <= st < inside_end: every lane is inside the matrix
        const int mc = mark_col - col0;          // the last marked column, in steps of lane 0
        int st = 0;
        slow_until(st, min(32, nsteps), one, four);
        if (MODE == kPB) {
            fast_until<true>(st, inside_end, one, four);
        } else if (MODE == kP2) {
            if (mc >= 0) {
                // columns below |left| - 2: an alignment ending there fails the span test whatever its tend, so only the
                // running maximum matters; it is folded into the tracked class once, marked as "ended too early"
                const int zs = max(mc - 2, 0);
                const int before = st;
                fast_until<false>(st, min(inside_end, (zs >> 4) << 4), one, four);
                if (st != before) {
                    const u32 nb = __vmaxu2(bestc, best | kOnes);
                    const u32 x = nb ^ bestc;
                    bestc = nb;
                    if (x > 0xffffu) { st_hi = lane; raw_hi = 0; }       // column 0: tend = 1
                    if (x & 0xffffu) { st_lo = lane; raw_lo = 0; }
                }
                // the lanes pass the kept column and the last marked column: guarded steps (the guard-free body with
                // those two checks unrolled four times measured slower here, unlike in the junction zone below)
                slow_until(st, min(nsteps, ((mc + 32 + 15) >> 4) << 4), one, four);
            }
            if (MULTI) {
                fast_until<true>(st, inside_end, one, four);
            } else {
                // Dominance exit (DESIGN.md section 4.9).  Right of |left| the template repeats with period m and the
                // DP is max-plus, so if the cut at step s is <= the cut at step s - P (P a multiple of m and of 16, both
                // cuts wholly right of the last marked column) every later cell is <= one P columns to its left that
                // was already folded into the record; only a strictly higher class replaces the record, so it is final.
                // Checks every P steps from the trip at which lane 31 reaches check_col (and has passed mark_col).
                next_check = -1;
                if (exits && mc >= 0) {
                    const int c0 = max(st, ((check_col - col0 + 32 + 15) >> 4) << 4);
                    if (c0 + period < inside_end) next_check = c0;
                    __stcg(kept_io + lane, 0u); __stcg(kept_io + 32 + lane, 0u); __stcg(kept_io + 64 + lane, 0u);
                    __stcg(kept_io + 96 + lane, (u32)period);
                }
                fast_until<true, false, true>(st, inside_end, one, four);
                if (exit_st >= 0) return;
            }
        } else {
            // plain steps up to the first junction / marked column, then guard-free steps that look for both
            const int first = min(zone_start, mc >= 0 ? mc : zone_start);
            fast_until<true>(st, min(inside_end, (first >> 4) << 4), one, four);
            if (MULTI && late_pending && st + 16 <= inside_end) late_load();      // the guard-free zone steps follow
            fast_until<true, true>(st, inside_end, one, four);
        }
        slow_until(st, nsteps, one, four);
    }
};

// round 3: 512 bases.  Shared memory per warp: the profile (2 KB per four rows) + the junction vectors as three 4-byte
// planes (384 bytes per row): 14 KB at R = 16, 224 KB for the 16 warps of a block
constexpr int kMaxRPair3 = 16;
constexpr int kMaxRPair2 = kMaxRPair3;   // round 2 pairs the same reads, so that round 3 can resume from its state
constexpr int kPairEntry = 1 << 30;      // order[] entry of a long pair's stripe: (index into pairs[] << 7) | code, this bit set

__host__ __device__ __forceinline__ int pair_rows(int q_len) {
    int R = (q_len + 31) / 32;
    return R < kMinR ? kMinR : R;
}

// Work distribution of the fused launches.  Items: the batch's 32-bit entries [0, n_rest) (in dependency order), then
// its pairs.  A long-read stripe is a latency-bound chain; next to three warps that saturate the DPX pipe it crawls at
// a fraction of its speed and becomes the kernel's tail.  So the 32-bit entries are dealt block-major: they fill whole
// blocks (four such warps per scheduler overlap each other's latencies), the other blocks start on pairs at once
// (slot-major, so a small batch spreads over the SMs), and everything left is pulled in order from *counter.
struct Deal {          // computed by the host, read from the kernel's parameter bank (no registers held across a task)
    int n_rest, n_pairs;
    int static_rest;   // 32-bit entries dealt block-major to blocks [0, nb_long)
    int nb_long;
    int static_pairs;  // pairs dealt slot-major to the other blocks
};
__host__ __device__ inline Deal make_deal(int n_rest, int n_pairs, int wpb, int grid) {
    Deal d;
    d.n_rest = n_rest; d.n_pairs = n_pairs;
    d.static_rest = n_rest < wpb * grid ? n_rest : wpb * grid;
    d.nb_long = (d.static_rest + wpb - 1) / wpb;
    const int room = wpb * (grid - d.nb_long);
    d.static_pairs = n_pairs < room ? n_pairs : room;
    return d;
}
// next item: < n_rest: entry of the 32-bit kernels; else pair (item - n_rest); -1: done
__device__ __forceinline__ int next_item(const Deal& dl, bool& first, int* counter) {
    if (dl.nb_long < 0) {       // plain dealing: one slot-major round over all items, then dynamic pulls
        const int n = dl.n_rest + dl.n_pairs;
        if (first) {
            first = false;
            const int i = (threadIdx.x >> 5) * (int)gridDim.x + (int)blockIdx.x;
            return i < n ? i : -1;
        }
        int i = 0;
        if ((threadIdx.x & 31) == 0) i = atomicAdd(counter, 1);
        i = __shfl_sync(kFull, i, 0) + (blockDim.x >> 5) * (int)gridDim.x;
        return i < n ? i : -1;
    }
    if (first) {
        first = false;
        const int wpb = blockDim.x >> 5, warp = threadIdx.x >> 5, blk = (int)blockIdx.x;
        if (blk < dl.nb_long) {
            const int e = blk * wpb + warp;
            if (e < dl.static_rest) return e;
        } else {
            const int p = warp * ((int)gridDim.x - dl.nb_long) + (blk - dl.nb_long);
            if (p < dl.static_pairs) return dl.n_rest + p;
        }
    }
    int d = 0;
    if ((threadIdx.x & 31) == 0) d = atomicAdd(counter, 1);
    d = __shfl_sync(kFull, d, 0);
    const int rest_left = dl.n_rest - dl.static_rest;
    if (d < rest_left) return dl.static_rest + d;
    const int p = dl.static_pairs + d - rest_left;
    return p < dl.n_pairs ? dl.n_rest + p : -1;
}

// ---- round 2 -------------------------------------------------------------------------------------------------------
template <int R>
__device__ __forceinline__ void pair2_task(const Pair2& pt, const Task* __restrict__ tasks, const uint32_t* __restrict__ pool,
                                           uint4* prof, int lane, u32 one, unsigned four, int4* out, u32* state,
                                           unsigned long long* skipped, u32* kept) {
    const Task ta = tasks[pt.a];
    Task tb = ta;
    int q_b = 0;
    if (pt.b >= 0) { tb = tasks[pt.b]; q_b = tb.q_len; }
    __syncwarp();
    build_profile<R>(prof, pool + ta.q_word, ta.q_len, pool + tb.q_word, q_b, lane * R, lane, false);
    __syncwarp();
    Sweep<R, kP2> sw;
    sw.prof = prof; sw.twords = pool + ta.t_word; sw.t_len = ta.t_len; sw.lane = lane;
    sw.mark_col = pt.mark_col;
    sw.col0 = 0; sw.resume = nullptr;
    sw.save_col = pt.mark_col - 2;
    sw.save = (state && pt.state_off >= 0 && sw.save_col >= 0) ? state + (size_t)pt.state_off * 32 : nullptr;
    sw.exits = pt.check_col >= 0;
    sw.check_col = pt.check_col; sw.period = pt.period;
    sw.kept_io = kept + (size_t)((blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 128);
    sw.run(one, four, 0);
    if (sw.exit_st >= 0 && lane == 0) {
        // lane l swept exit_st - l columns instead of t_len
        const unsigned long long cols32 = 32ull * (unsigned)ta.t_len - (32ull * (unsigned)sw.exit_st - 496ull);
        atomicAdd(&skipped[0], (unsigned long long)R * cols32);
        atomicAdd(&skipped[1], (unsigned long long)(ta.q_len + q_b) * cols32);
    }
    // per half: (score, smallest end column, mark of the best word there) -> one 32-bit key, warp maximum
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const u32 cls = half ? (sw.bestc & 0xffffu) : (sw.bestc >> 16);
        const u32 raw = half ? (sw.raw_lo & 0xffffu) : (sw.raw_hi >> 16);
        const int st = half ? sw.st_lo : sw.st_hi;
        const int score = (int)(cls - (kBias + 1)) >> 1;
        const int col = st - lane;
        unsigned key = 0;
        if (score > 0) key = ((unsigned)score << 17) | ((0xffffu - (unsigned)col) << 1) | (raw & 1u);
        key = __reduce_max_sync(kFull, key);
        const int tid = half ? pt.b : pt.a;
        if (lane == 0 && tid >= 0) {
            int4 rec = make_int4(0, 0, 0, 0);
            if (key) {
                const int c = 0xffff - (int)((key >> 1) & 0xffffu);
                const bool inside = c <= pt.mark_col || !(key & 1u);
                rec = make_int4((int)(key >> 17), inside ? 0 : pt.mark_col + 1, c + 1, 0);
            }
            out[tid] = rec;
        }
    }
}

// One stripe of a pair of long reads in round 2.  pt.state_off = index of the pair's CoopInfo; the pair's flag words:
// [2S] stripes done, [2S + 2] / [2S + 3] best key of read A / read B over the stripes done so far.
template <int R>
__device__ __noinline__ void pair2_stripe(const Pair2& pt, int s, const Task* __restrict__ tasks, const uint32_t* __restrict__ pool,
                                          const RestArgs& ra, uint4* prof, int lane, u32 one, unsigned four, int4* out) {
    const CoopInfo ci = ra.coop[pt.state_off];
    const int S = ci.n_stripes;
    int* F = ra.flags + ci.flag_off;
    ulonglong2* bnd_a = reinterpret_cast<ulonglong2*>(ra.scratch + ci.data_off);
    ulonglong2* bnd_b = bnd_a + ci.bnd_stride;
    const Task ta = tasks[pt.a];
    Task tb = ta;
    int q_b = 0;
    if (pt.b >= 0) { tb = tasks[pt.b]; q_b = tb.q_len; }
    __syncwarp();
    build_profile<R>(prof, pool + ta.q_word, ta.q_len, pool + tb.q_word, q_b, s * 32 * R + lane * R, lane, false);
    __syncwarp();
    Sweep<R, kP2, true> sw;
    sw.prof = prof; sw.twords = pool + ta.t_word; sw.t_len = ta.t_len; sw.lane = lane;
    sw.mark_col = pt.mark_col;
    sw.col0 = 0; sw.resume = nullptr; sw.save = nullptr; sw.save_col = -1;
    sw.top = s > 0; sw.bot = s + 1 < S;
    sw.bnd_in = (s & 1) ? bnd_a : bnd_b; sw.bnd_out = (s & 1) ? bnd_b : bnd_a;
    sw.tag_in = stripe_tag(ra.epoch, s - 1); sw.tag_out = stripe_tag(ra.epoch, s); sw.spin = ra.spin;
    sw.run(one, four, 0);
    unsigned keys[2];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const u32 cls = half ? (sw.bestc & 0xffffu) : (sw.bestc >> 16);
        const u32 raw = half ? (sw.raw_lo & 0xffffu) : (sw.raw_hi >> 16);
        const int st = half ? sw.st_lo : sw.st_hi;
        const int score = (int)(cls - (kBias + 1)) >> 1;
        unsigned key = 0;
        if (score > 0) key = ((unsigned)score << 17) | ((0xffffu - (unsigned)(st - lane)) << 1) | (raw & 1u);
        keys[half] = __reduce_max_sync(kFull, key);
    }
    if (lane == 0) {
        unsigned* K = reinterpret_cast<unsigned*>(F + 2 * S + 2);
        atomicMax(&K[0], keys[0]);
        atomicMax(&K[1], keys[1]);
        __threadfence();
        if (atomicAdd(F + 2 * S, 1) == S - 1) {
            __threadfence();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int tid = half ? pt.b : pt.a;
                if (tid < 0) continue;
                const unsigned key = atomicMax(&K[half], 0u);
                int4 rec = make_int4(0, 0, 0, 0);
                if (key) {
                    const int c = 0xffff - (int)((key >> 1) & 0xffffu);
                    const bool inside = c <= pt.mark_col || !(key & 1u);
                    rec = make_int4((int)(key >> 17), inside ? 0 : pt.mark_col + 1, c + 1, 0);
                }
                out[tid] = rec;
            }
        }
    }
}

template <int R>
__device__ __forceinline__ void pair2_stripe_dispatch(int r, const Pair2& pt, int s, const Task* __restrict__ tasks,
                                                      const uint32_t* __restrict__ pool, const RestArgs& ra, uint4* prof, int lane,
                                                      u32 one, unsigned four, int4* out) {
    if constexpr (is_coop_height(R))
        if (r == R) { pair2_stripe<R>(pt, s, tasks, pool, ra, prof, lane, one, four, out); return; }
    if constexpr (R < kMaxRLadder) pair2_stripe_dispatch<R + 1>(r, pt, s, tasks, pool, ra, prof, lane, one, four, out);
}

template <int R>
__device__ __forceinline__ void pair2_dispatch(int r, const Pair2& pt, const Task* __restrict__ tasks,
                                               const uint32_t* __restrict__ pool, uint4* prof, int lane, u32 one,
                                               unsigned four, int4* out, u32* state, unsigned long long* skipped, u32* kept) {
    if (r == R) { pair2_task<R>(pt, tasks, pool, prof, lane, one, four, out, state, skipped, kept); return; }
    if constexpr (R < kMaxRPair2) pair2_dispatch<R + 1>(r, pt, tasks, pool, prof, lane, one, four, out, state, skipped, kept);
}

// Round 2: the batch's 32-bit entries (stripes of long reads first: they are the critical path) and then its pairs, one
// persistent launch.  out[task] = (score, 0 if the alignment starts at a column <= |left| else |left| + 1, tend, 0) for
// paired tasks, the exact (score, tstart, tend, 0) for the others.
#ifdef NR_DEFINE_PAIR_ROUND2_KERNEL      // defined by the one translation unit that owns this kernel (nr_launch_pair2.cu)
__global__ void __launch_bounds__(32 * kWarpsPerBlock, 1)
pair_round2_kernel(const Pair2* __restrict__ pairs, Deal dl, const Task* __restrict__ tasks, RestArgs ra,
                   const uint32_t* __restrict__ pool, ScoreW scw, int* counter, int smem_stride, int4* out, u32* state,
                   u32* kept) {
    extern __shared__ uint4 psmem[];
    const ScoreView<true> sc(scw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint4* prof = psmem + warp * smem_stride;
    bool first = true;
    for (;;) {
        const int i = next_item(dl, first, counter);
        if (i < 0) break;
        if (i < ra.n_order) {
            const int e = ra.order[i];
            if (e & kPairEntry) {           // a stripe of a pair of long reads: (pair index << 7) | (1 + stripe)
                const Pair2 mp = pairs[(e & ~kPairEntry) >> kCodeBits];
                pair2_stripe_dispatch<kMinR>(ra.coop[mp.state_off].rows, mp, (e & ((1 << kCodeBits) - 1)) - 1, tasks, pool, ra, prof, lane,
                                             (u32)sc.one, sc.four, out);
            } else {
                exact_entry(e, tasks, pool, sc, ra, reinterpret_cast<int4*>(prof), lane, out);
            }
            continue;
        }
        const Pair2 pt = pairs[i - ra.n_order];
        int q = tasks[pt.a].q_len;
        if (pt.b >= 0) q = max(q, tasks[pt.b].q_len);
        pair2_dispatch<kMinR>(pair_rows(q), pt, tasks, pool, prof, lane, (u32)sc.one, sc.four, out, state,
                              reinterpret_cast<unsigned long long*>(counter + kExitSlot), kept);
    }
}
#endif

// ---- round 3 -------------------------------------------------------------------------------------------------------
// One rung of one read from the (P, J) tokens: score, "ends in right", and the mark of the best non-prefix candidate.
__device__ __forceinline__ void rung_of(u32 P, u32 J, u32 rc, int& score, bool& in_right, bool& unmarked) {
    const u32 np = max(J, rc);
    const int s_p = (int)(P - kBias) >> 1;
    const int s_np = (int)(np - 2 * kBias) >> 1;
    in_right = s_np > s_p;
    score = max(s_p, s_np);
    unmarked = np & 1u;
}

// The per-read selection over a pair's rung tokens (nanoRepeat_bam.py:423-431); reads whose result hinges on a tie the
// 16-bit words cannot order are appended to redo[] (entries of ladder_kernel's order[]; long pairs: task indices for
// the host, see nr_api.cu).
__device__ __forceinline__ void pair3_select(const Pair3& pt, const LadderTask& ta, const LadderTask& tb, int kmin, u32 rcand,
                                             const uint2* rungs, int lane, int min_score, int4* sel, int* redo_count, int32_t* redo,
                                             int redo_shift) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int tid = half ? pt.b : pt.a;
        if (tid < 0) continue;
        const LadderTask& tk = half ? tb : ta;
        const u32 rc = half ? (rcand & 0xffffu) : (rcand >> 16);
        int top = 0;
        for (int k = tk.kmin + lane; k <= tk.kmax; k += 32) {
            const uint2 t = rungs[k - kmin];
            int s; bool ir, um;
            rung_of(half ? (t.x & 0xffffu) : (t.x >> 16), half ? (t.y & 0xffffu) : (t.y >> 16), rc, s, ir, um);
            if (s >= min_score) top = max(top, s);
        }
        top = __reduce_max_sync(kFull, top);
        int n = 0, sum = 0, unsure = 0;
        if (top > 0) {
            for (int k = tk.kmin + lane; k <= tk.kmax; k += 32) {
                const uint2 t = rungs[k - kmin];
                int s; bool ir, um;
                rung_of(half ? (t.x & 0xffffu) : (t.x >> 16), half ? (t.y & 0xffffu) : (t.y >> 16), rc, s, ir, um);
                if (s == top && ir) {
                    if (um) unsure = 1;
                    else { ++n; sum += k; }
                }
            }
        }
        n = __reduce_add_sync(kFull, n);
        sum = __reduce_add_sync(kFull, sum);
        unsure = __any_sync(kFull, unsure);
        if (lane == 0) {
            sel[tk.read] = make_int4(top, n, sum, 0);
            if (unsure) redo[atomicAdd(redo_count, 1)] = tid << redo_shift;
        }
    }
}

template <int R>
__device__ __forceinline__ void pair3_task(const Pair3& pt, const LadderTask* __restrict__ tasks,
                                           const uint32_t* __restrict__ qpool, const uint32_t* __restrict__ pool,
                                           const LadderRegion* __restrict__ regs, uint4* prof, int lane, u32 one,
                                           unsigned four, int min_score, uint2* prung, int4* sel, int* redo_count,
                                           int32_t* redo, const u32* __restrict__ qstate) {
    // either half may be absent (a read round 2 gave no size keeps its place in a resumed pair)
    const bool ha = pt.a >= 0, hb = pt.b >= 0;
    const LadderTask tv = tasks[ha ? pt.a : pt.b];
    LadderTask ta = tv, tb = tv;
    int q_a = 0, q_b = 0;
    if (ha) { ta = tasks[pt.a]; q_a = ta.q_len; }
    if (hb) { tb = tasks[pt.b]; q_b = tb.q_len; }
    const LadderRegion reg = regs[tv.region];
    const int kmin = (ha && hb) ? min(ta.kmin, tb.kmin) : tv.kmin;
    const int kmax = (ha && hb) ? max(ta.kmax, tb.kmax) : tv.kmax;
    u32* bsm = reinterpret_cast<u32*>(prof + StripeCfg<R>::PROF_INT4);
    uint2* rungs = prung + pt.rung_off;
    __syncwarp();
    build_profile<R>(prof, qpool + ta.q_word, q_a, qpool + tb.q_word, q_b, lane * R, lane, true);
    __syncwarp();
    u32 rcand;
    {
        Sweep<R, kPB> sw;
        sw.prof = prof; sw.twords = pool + reg.rev_word; sw.t_len = reg.n_right; sw.lane = lane;
        sw.mark_col = -1; sw.q_a = q_a; sw.q_b = q_b;
        sw.col0 = 0; sw.resume = nullptr; sw.save = nullptr; sw.save_col = -1;
        sw.run(one, four, 0);
        const u32 ra = __reduce_max_sync(kFull, sw.best >> 16), rb = __reduce_max_sync(kFull, sw.best & 0xffffu);
        rcand = pk2((int)ra + kBias + 1, (int)rb + kBias + 1);      // forward part empty: score 0, unmarked
        sw.store_junction_vectors(reinterpret_cast<u32*>(prof), bsm);
    }
    __syncwarp();
    build_profile<R>(prof, qpool + ta.q_word, q_a, qpool + tb.q_word, q_b, lane * R, lane, false);
    __syncwarp();
    {
        Sweep<R, kPF> sw;
        sw.prof = prof; sw.twords = pool + reg.fwd_word; sw.t_len = reg.n_left + reg.m * kmax; sw.lane = lane;
        sw.mark_col = reg.n_left - 1; sw.bsm = bsm; sw.rung_out = rungs;
        sw.m = reg.m; sw.jnext = reg.n_left + reg.m * kmin; sw.kcnt = 0;
        sw.save = nullptr; sw.save_col = -1;
        const bool resumes = qstate && pt.state_off >= 0;
        sw.col0 = resumes ? reg.n_left - 1 : 0;
        sw.resume = resumes ? qstate + (size_t)pt.state_off * 32 : nullptr;
        sw.run(one, four, sw.jnext - 1 - sw.col0);
    }
    __syncwarp();
    pair3_select(pt, ta, tb, kmin, rcand, rungs, lane, min_score, sel, redo_count, redo, kCodeBits);
}

// Long pairs in round 3.  pt.pad[0] = the pair's CoopInfo; scratch (int4 units from ci.data_off): boundary rows a, b of the
// backward sweep | a, b of the forward sweep | the backward stripes' junction state, 3 planes of ci.b_stride words |
// token rows a, b.  Flag words: [2S] backward stripes done, [2S + 2] / [2S + 3] the R-only best of read A / read B.
template <int R>
__device__ __noinline__ void pair3_bwd_stripe(const Pair3& pt, int s, const LadderTask* __restrict__ tasks,
                                              const uint32_t* __restrict__ qpool, const uint32_t* __restrict__ pool,
                                              const LadderRegion* __restrict__ regs, const RestArgs& ra, uint4* prof, int lane,
                                              u32 one, unsigned four) {
    const CoopInfo ci = ra.coop[pt.pad[0]];
    const int S = ci.n_stripes;
    int* F = ra.flags + ci.flag_off;
    ulonglong2* bnd_a = reinterpret_cast<ulonglong2*>(ra.scratch + ci.data_off);
    ulonglong2* bnd_b = bnd_a + ci.bnd_stride;
    u32* stage = reinterpret_cast<u32*>(ra.scratch + ci.data_off + 4 * ci.bnd_stride);
    const LadderTask ta = tasks[pt.a], tb = tasks[pt.b];
    const LadderRegion reg = regs[ta.region];
    __syncwarp();
    build_profile<R>(prof, qpool + ta.q_word, ta.q_len, qpool + tb.q_word, tb.q_len, s * 32 * R + lane * R, lane, true);
    __syncwarp();
    Sweep<R, kPB, true> sw;
    sw.prof = prof; sw.twords = pool + reg.rev_word; sw.t_len = reg.n_right; sw.lane = lane;
    sw.mark_col = -1; sw.q_a = ta.q_len; sw.q_b = tb.q_len;
    sw.col0 = 0; sw.resume = nullptr; sw.save = nullptr; sw.save_col = -1;
    sw.top = s > 0; sw.bot = s + 1 < S;
    sw.bnd_in = (s & 1) ? bnd_a : bnd_b; sw.bnd_out = (s & 1) ? bnd_b : bnd_a;
    sw.tag_in = stripe_tag(ra.epoch, s - 1); sw.tag_out = stripe_tag(ra.epoch, s); sw.spin = ra.spin;
    sw.run(one, four, 0);
    sw.store_stage(stage, ci.b_stride, s * 32 * R);
    const u32 ba = __reduce_max_sync(kFull, sw.best >> 16), bb = __reduce_max_sync(kFull, sw.best & 0xffffu);
    __syncwarp();                       // every lane's junction state is stored
    if (lane == 0) {
        unsigned* K = reinterpret_cast<unsigned*>(F + 2 * S + 2);
        atomicMax(&K[0], ba);
        atomicMax(&K[1], bb);
        __threadfence();
        atomicAdd(F + 2 * S, 1);
    }
}

template <int R>
__device__ __noinline__ void pair3_fwd_stripe(const Pair3& pt, int s, const LadderTask* __restrict__ tasks,
                                              const uint32_t* __restrict__ qpool, const uint32_t* __restrict__ pool,
                                              const LadderRegion* __restrict__ regs, const RestArgs& ra, uint4* prof, int lane,
                                              u32 one, unsigned four, int min_score, uint2* prung, int4* sel, int* redo_count,
                                              int32_t* redo) {
    const CoopInfo ci = ra.coop[pt.pad[0]];
    const int S = ci.n_stripes;
    int* F = ra.flags + ci.flag_off;
    ulonglong2* bnd_a = reinterpret_cast<ulonglong2*>(ra.scratch + ci.data_off + 2 * ci.bnd_stride);
    ulonglong2* bnd_b = bnd_a + ci.bnd_stride;
    const u32* stage = reinterpret_cast<const u32*>(ra.scratch + ci.data_off + 4 * ci.bnd_stride);
    ulonglong2* tok_a = reinterpret_cast<ulonglong2*>(ra.scratch + ci.data_off + 4 * ci.bnd_stride + (3 * ci.b_stride + 3) / 4);
    ulonglong2* tok_b = tok_a + ci.tok_stride;
    const LadderTask ta = tasks[pt.a], tb = tasks[pt.b];
    const LadderRegion reg = regs[ta.region];
    const int kmin = min(ta.kmin, tb.kmin), kmax = max(ta.kmax, tb.kmax);
    u32* bsm = reinterpret_cast<u32*>(prof + StripeCfg<R>::PROF_INT4);
    uint2* rungs = prung + pt.rung_off;
    __syncwarp();
    build_profile<R>(prof, qpool + ta.q_word, ta.q_len, qpool + tb.q_word, tb.q_len, s * 32 * R + lane * R, lane, false);
    __syncwarp();
    Sweep<R, kPF, true> sw;
    sw.prof = prof; sw.twords = pool + reg.fwd_word; sw.t_len = reg.n_left + reg.m * kmax; sw.lane = lane;
    sw.mark_col = reg.n_left - 1; sw.bsm = bsm; sw.bsm_w = bsm; sw.rung_out = rungs;
    sw.m = reg.m; sw.jnext = reg.n_left + reg.m * kmin; sw.kcnt = 0;
    sw.q_a = ta.q_len; sw.q_b = tb.q_len;
    sw.save = nullptr; sw.save_col = -1; sw.col0 = 0; sw.resume = nullptr;
    sw.top = s > 0; sw.bot = s + 1 < S;
    sw.bnd_in = (s & 1) ? bnd_a : bnd_b; sw.bnd_out = (s & 1) ? bnd_b : bnd_a;
    sw.tok_in = (s & 1) ? tok_a : tok_b; sw.tok_out = (s & 1) ? tok_b : tok_a;
    sw.tag_in = stripe_tag(ra.epoch, s - 1); sw.tag_out = stripe_tag(ra.epoch, s); sw.spin = ra.spin;
    sw.bstage = stage; sw.b_stride = ci.b_stride; sw.brow0 = s * 32 * R;
    sw.bdone = F + 2 * S; sw.bdone_need = S;
    sw.run(one, four, sw.jnext - 1);
    if (s == S - 1) {
        // the last rows finalised every rung: the selection of both reads (the R-only class from the backward stripes,
        // which are all done: this stripe waited for them before its first junction column)
        __syncwarp();
        if (sw.late_pending) wait_cols(sw.bdone, sw.bdone_need, lane, ra.spin);
        const unsigned* K = reinterpret_cast<const unsigned*>(F + 2 * S + 2);
        const u32 rcand = pk2((int)__ldcg(&K[0]) + kBias + 1, (int)__ldcg(&K[1]) + kBias + 1);
        pair3_select(pt, ta, tb, kmin, rcand, rungs, lane, min_score, sel, ra.redo_long_count, ra.redo_long, 0);
    }
}

template <int R>
__device__ __forceinline__ void pair3_stripe_dispatch(int r, const Pair3& pt, int code, const LadderTask* __restrict__ tasks,
                                                      const uint32_t* __restrict__ qpool, const uint32_t* __restrict__ pool,
                                                      const LadderRegion* __restrict__ regs, const RestArgs& ra, uint4* prof,
                                                      int lane, u32 one, unsigned four, int min_score, uint2* prung, int4* sel,
                                                      int* redo_count, int32_t* redo) {
    if constexpr (is_coop_height(R))
        if (r == R) {
            if (code < kCodeFwd) pair3_bwd_stripe<R>(pt, code - 1, tasks, qpool, pool, regs, ra, prof, lane, one, four);
            else pair3_fwd_stripe<R>(pt, code - kCodeFwd, tasks, qpool, pool, regs, ra, prof, lane, one, four, min_score, prung, sel,
                                     redo_count, redo);
            return;
        }
    if constexpr (R < kMaxRLadder)
        pair3_stripe_dispatch<R + 1>(r, pt, code, tasks, qpool, pool, regs, ra, prof, lane, one, four, min_score, prung, sel, redo_count, redo);
}

template <int R>
__device__ __forceinline__ void pair3_dispatch(int r, const Pair3& pt, const LadderTask* __restrict__ tasks,
                                               const uint32_t* __restrict__ qpool, const uint32_t* __restrict__ pool,
                                               const LadderRegion* __restrict__ regs, uint4* prof, int lane, u32 one,
                                               unsigned four, int min_score, uint2* prung, int4* sel, int* redo_count,
                                               int32_t* redo, const u32* __restrict__ qstate) {
    if (r == R) { pair3_task<R>(pt, tasks, qpool, pool, regs, prof, lane, one, four, min_score, prung, sel, redo_count, redo, qstate); return; }
    if constexpr (R < kMaxRPair3)
        pair3_dispatch<R + 1>(r, pt, tasks, qpool, pool, regs, prof, lane, one, four, min_score, prung, sel, redo_count, redo, qstate);
}

// Round 3: the batch's 32-bit entries (stripes of long reads, reads without an anchor) and then its pairs, one
// persistent launch.  sel[read] = (top score, n tied rungs that span both flanks, sum of their k, 0); paired reads
// whose selection hinges on an undecidable tie go to redo[] (entries for ladder_kernel).
#ifdef NR_DEFINE_PAIR_LADDER_KERNEL      // defined by the one translation unit that owns this kernel (nr_launch_pair3.cu)
__global__ void __launch_bounds__(32 * kWarpsPerBlock, 1)
pair_ladder_kernel(const Pair3* __restrict__ pairs, Deal dl, const LadderTask* __restrict__ tasks, RestArgs ra,
                   const uint32_t* __restrict__ qpool, const uint32_t* __restrict__ pool,
                   const LadderRegion* __restrict__ regs, ScoreW scw, int* counter,
                   int smem_stride, uint2* prung, int4* out, int4* sel, int* redo_count, int32_t* redo,
                   const u32* __restrict__ qstate) {
    extern __shared__ uint4 psmem[];
    const ScoreView<true> sc(scw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint4* prof = psmem + warp * smem_stride;
    bool first = true;
    for (;;) {
        const int i = next_item(dl, first, counter);
        if (i < 0) break;
        if (i < ra.n_order) {
            const int e = ra.order[i];
            if (e & kPairEntry) {           // a stripe of a pair of long reads: (pair index << 7) | (1 + s backward, 64 + s forward)
                const Pair3 mp = pairs[(e & ~kPairEntry) >> kCodeBits];
                pair3_stripe_dispatch<kMinR>(mp.R, mp, e & ((1 << kCodeBits) - 1), tasks, qpool, pool, regs, ra, prof, lane, (u32)sc.one,
                                             sc.four, sc.min_score, prung, sel, redo_count, redo);
            } else {
                ladder_entry<true, kMaxRLadder>(e, tasks, qpool, pool, regs, sc, ra, reinterpret_cast<int4*>(prof), lane, out, sel);
            }
            continue;
        }
        const Pair3 pt = pairs[i - ra.n_order];
        int rows = pt.R;
        if (rows <= 0) {
            int q = pt.a >= 0 ? tasks[pt.a].q_len : 0;
            if (pt.b >= 0) q = max(q, tasks[pt.b].q_len);
            rows = pair_rows(q);
        }
        pair3_dispatch<kMinR>(rows, pt, tasks, qpool, pool, regs, prof, lane, (u32)sc.one, sc.four, sc.min_score, prung, sel, redo_count, redo, qstate);
    }
}
#endif

}  // namespace pr
}  // namespace nr
