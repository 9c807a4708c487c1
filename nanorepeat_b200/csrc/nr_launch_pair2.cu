// pair_round2_kernel: round 2 on u16x2 words, two reads per warp, plus the batch's 32-bit entries (nr_pair_kernels.cuh)
#define NR_DEFINE_PAIR_ROUND2_KERNEL
#include "nr_launch.h"
#include <mutex>
namespace nrl {
cudaError_t launch_pair_round2(int blocks, int threads, size_t smem, cudaStream_t st, const nr::pr::Pair2* pairs,
                               const nr::pr::Deal& deal, const nr::Task* tasks, const nr::RestArgs& ra, const uint32_t* pool,
                               const nr::ScoreW& k, int* counter, int stride, int4* out, uint32_t* state,
                               uint32_t* kept) {
    static std::mutex mu;
    static bool done = false;
    {
        std::lock_guard<std::mutex> lk(mu);
        cudaError_t e = prepare(nr::pr::pair_round2_kernel, done);
        if (e != cudaSuccess) return e;
    }
    nr::pr::pair_round2_kernel<<<blocks, threads, smem, st>>>(pairs, deal, tasks, ra, pool, k, counter, stride, out, state, kept);
    return cudaGetLastError();
}
}  // namespace nrl
