// anchor_pair_kernel: Step 1's anchor search on u16x2 words (nr_pair_kernels.cuh), host side in nr_anchor.cu.
//
// One warp per read strand: the strand is the template, the region's left and right anchor are the two queries, one
// per 16-bit half of every DP word, so one DPX instruction updates a cell of each anchor.  An anchor (up to
// --anchor_len = 1 000 bases) is longer than one paired stripe (32 * R rows), so the SAME warp sweeps the stripes of its
// pair one after the other; the bottom row of a stripe reaches the next one through a per-warp scratch row in global
// memory (L2), as the tagged boundary entries the stripes of a long round-2 pair hand down (Sweep<R, kP2, true>).  The
// entries of stripe s are all written before stripe s + 1 starts, so a tag check never waits.  The mark bit is inert
// (no marked column), so what a half yields is its key (score, smallest end column): the contract's (score, tend).
// No dominance exit: a read is not periodic.
#include "nr_launch_anchor.h"
#include <mutex>

namespace nr {
namespace pr {

// Per half: the best score and the first column reaching it, as one key (score << 17 | (0xffff - col) << 1 | 1)
template <int R>
__device__ __forceinline__ void half_keys(const Sweep<R, kP2, true>& sw, int lane, unsigned* keys) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const u32 cls = half ? (sw.bestc & 0xffffu) : (sw.bestc >> 16);
        const int st = half ? sw.st_lo : sw.st_hi;
        const int score = (int)(cls - (kBias + 1)) >> 1;
        unsigned key = 0;
        if (score > 0) key = ((unsigned)score << 17) | ((0xffffu - (unsigned)(st - lane)) << 1) | 1u;
        keys[half] = max(keys[half], __reduce_max_sync(kFull, key));
    }
}

template <int R>
__device__ __noinline__ void anchor_pair(const AnchorPair& p, const uint32_t* __restrict__ pool, uint4* prof, ulonglong2* bnd,
                                         size_t bnd_stride, int lane, u32 one, unsigned four, int* spin, uint2* out) {
    const uint32_t* qa = pool + p.qa_word;
    const uint32_t* qb = p.q_b > 0 ? pool + p.qb_word : qa;
    unsigned keys[2] = {0u, 0u};
    for (int s = 0; s < p.S; ++s) {
        __syncwarp();
        build_profile<R>(prof, qa, p.q_a, qb, p.q_b, s * 32 * R + lane * R, lane, false);
        __syncwarp();
        Sweep<R, kP2, true> sw;
        sw.prof = prof; sw.twords = pool + p.t_word; sw.t_len = p.t_len; sw.lane = lane;
        sw.mark_col = -1;                    // no marked column: every word stays unmarked
        sw.col0 = 0; sw.resume = nullptr; sw.save = nullptr; sw.save_col = -1;
        sw.top = s > 0; sw.bot = s + 1 < p.S;
        sw.bnd_in = bnd + ((s + 1) & 1) * bnd_stride; sw.bnd_out = bnd + (s & 1) * bnd_stride;
        sw.tag_in = stripe_tag(1, s - 1); sw.tag_out = stripe_tag(1, s); sw.spin = spin;
        sw.run(one, four, 0);
        half_keys<R>(sw, lane, keys);
        __syncwarp();
        __threadfence_block();               // the next stripe's lanes read what lane 31 wrote
    }
    if (lane == 0) *out = make_uint2(keys[0], keys[1]);
}

template <int R>
__device__ __forceinline__ void anchor_dispatch(int r, const AnchorPair& p, const uint32_t* __restrict__ pool, uint4* prof,
                                                ulonglong2* bnd, size_t bnd_stride, int lane, u32 one, unsigned four, int* spin,
                                                uint2* out) {
    if constexpr (is_coop_height(R))
        if (r == R) { anchor_pair<R>(p, pool, prof, bnd, bnd_stride, lane, one, four, spin, out); return; }
    if constexpr (R < kMaxRPair2) anchor_dispatch<R + 1>(r, p, pool, prof, bnd, bnd_stride, lane, one, four, spin, out);
}

// pairs in the order the host dealt them (longest first); keys[p.out] = (left key, right key); counter[0]: next pair,
// counter[1]: the give-up flag of the boundary waits (never raised: every entry is written before it is read)
__global__ void __launch_bounds__(32 * kWarpsPerBlock, 1)
anchor_pair_kernel(const AnchorPair* __restrict__ pairs, int n_pairs, const uint32_t* __restrict__ pool, ulonglong2* scratch,
                   size_t bnd_stride, int* counter, u32 one, unsigned four, uint2* keys) {
    extern __shared__ uint4 asmem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint4* prof = asmem + warp * StripeCfg<kMaxRPair2>::PROF_INT4;
    ulonglong2* bnd = scratch + (size_t)(blockIdx.x * (blockDim.x >> 5) + warp) * 2 * bnd_stride;
    for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(counter, 1);
        i = __shfl_sync(kFull, i, 0);
        if (i >= n_pairs) break;
        const AnchorPair p = pairs[i];
        anchor_dispatch<kMinR>(p.R, p, pool, prof, bnd, bnd_stride, lane, one, four, counter + 1, keys + p.out);
    }
}

}  // namespace pr
}  // namespace nr

namespace nrl {
size_t anchor_smem_bytes() { return sizeof(uint4) * nr::kWarpsPerBlock * nr::StripeCfg<nr::pr::kMaxRPair2>::PROF_INT4; }

cudaError_t launch_anchor_pairs(int blocks, cudaStream_t st, const nr::pr::AnchorPair* pairs, int n_pairs, const uint32_t* pool,
                                ulonglong2* scratch, size_t bnd_stride, int* counter, uint2* keys) {
    static std::mutex mu;
    static bool done = false;
    {
        std::lock_guard<std::mutex> lk(mu);
        cudaError_t e = prepare(nr::pr::anchor_pair_kernel, done);
        if (e != cudaSuccess) return e;
    }
    nr::pr::anchor_pair_kernel<<<blocks, 32 * nr::kWarpsPerBlock, anchor_smem_bytes(), st>>>(pairs, n_pairs, pool, scratch, bnd_stride,
                                                                                            counter, 1u, 4u, keys);
    return cudaGetLastError();
}
}  // namespace nrl
