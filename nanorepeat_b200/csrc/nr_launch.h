// nr_launch.h -- host-callable launchers of the kernels, one translation unit per kernel family so that the four
// families compile side by side (each is minutes of ptxas time) and a change to the host code does not rebuild them.
// Every launcher sets its kernel's shared-memory attributes once (maximum dynamic shared memory, carve-out all the way
// to shared: batches are launched from several host threads, a per-launch value set by one could fail another's launch)
// and returns the launch's cudaError_t.
#pragma once
#include "nr_kernels.cuh"
#include "nr_pair_kernels.cuh"

namespace nrl {

constexpr size_t kMaxDynShared = (size_t)nr::kWarpsPerBlock * 14 * 1024;   // 16 warps x 14 KB (paired ladder at R = 16): 224 of 227 KB

cudaError_t launch_exact(bool fixed, int blocks, int threads, size_t smem, cudaStream_t st, const nr::Task* tasks,
                         const nr::RestArgs& ra, const uint32_t* pool, const nr::ScoreW& k, int* counter, int stride, int4* out);
cudaError_t launch_ladder(bool flag, int blocks, int threads, size_t smem, cudaStream_t st, const nr::LadderTask* tasks,
                          const nr::RestArgs& ra, const int* n_order_dev, const uint32_t* qpool, const uint32_t* pool,
                          const nr::LadderRegion* regs, const nr::ScoreW& k, int* counter, int stride, int4* out, int4* sel);
cudaError_t launch_pair_round2(int blocks, int threads, size_t smem, cudaStream_t st, const nr::pr::Pair2* pairs,
                               const nr::pr::Deal& deal, const nr::Task* tasks, const nr::RestArgs& ra, const uint32_t* pool,
                               const nr::ScoreW& k, int* counter, int stride, int4* out, uint32_t* state,
                               uint32_t* kept);
cudaError_t launch_pair_ladder(int blocks, int threads, size_t smem, cudaStream_t st, const nr::pr::Pair3* pairs,
                               const nr::pr::Deal& deal, const nr::LadderTask* tasks, const nr::RestArgs& ra,
                               const uint32_t* qpool, const uint32_t* pool, const nr::LadderRegion* regs, const nr::ScoreW& k,
                               int* counter, int stride, uint2* prung, int4* out, int4* sel, int* redo_count, int32_t* redo,
                               const uint32_t* qstate);

// once per kernel function, thread-safe
template <class F>
inline cudaError_t prepare(F fn, bool& done) {
    if (done) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynShared);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e == cudaSuccess) done = true;
    return e;
}

}  // namespace nrl
