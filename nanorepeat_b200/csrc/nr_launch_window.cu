// window_kernel, ladder_bwd_kernel, ladder_fwd_kernel: the joint path (nr_window_kernel.cuh, nr_window_ladder.cuh), host
// side in nr_joint.cu.
#include "nr_window_ladder.cuh"
#include <mutex>

namespace nrl {
namespace {

// A kernel's maximum dynamic shared memory, set on its first launch (batches are launched from several host threads)
struct SmemOnce {
    std::once_flag once;
    cudaError_t err = cudaSuccess;
    template <class F>
    cudaError_t operator()(F fn, size_t bytes) {
        std::call_once(once, [&]() { err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); });
        return err;
    }
};

constexpr size_t kSmemSweep = (size_t)nrw::kWarps * 8 * nrw::kRows * sizeof(int);                       // window, backward
constexpr size_t kSmemFwd = (size_t)nrw::kWarps * (11 * nrw::kRows + 2 * nrw::kMaxK2) * sizeof(int);

}  // namespace

cudaError_t launch_window(int blocks, cudaStream_t st, const nrw::WinTask* tasks, int n_tasks, const uint32_t* pool,
                          const nrw::WinScore& sc, int4* scratch, int scratch_stride, int* counter, int2* out) {
    static SmemOnce attr;
    if (cudaError_t e = attr(nrw::window_kernel, kSmemSweep)) return e;
    nrw::window_kernel<<<blocks, 32 * nrw::kWarps, kSmemSweep, st>>>(tasks, n_tasks, pool, sc, scratch, scratch_stride, counter, out);
    return cudaGetLastError();
}

cudaError_t launch_ladder_bwd(int blocks, cudaStream_t st, const nrw::LadBwdTask* tasks, int n_tasks, const uint32_t* pool,
                              const nrw::WinScore& sc, int4* scratch, int scratch_stride, int* counter, int* bvec, int* ronly) {
    static SmemOnce attr;
    if (cudaError_t e = attr(nrw::ladder_bwd_kernel, kSmemSweep)) return e;
    nrw::ladder_bwd_kernel<<<blocks, 32 * nrw::kWarps, kSmemSweep, st>>>(tasks, n_tasks, pool, sc, scratch, scratch_stride, counter,
                                                                       bvec, ronly);
    return cudaGetLastError();
}

cudaError_t launch_ladder_fwd(int blocks, cudaStream_t st, const nrw::LadFwdTask* tasks, int n_tasks, const nrw::LadBwdTask* btasks,
                              const uint32_t* pool, const nrw::WinScore& sc, int4* scratch, int scratch_stride, int* counter,
                              const int* bvec, const int* ronly, int* cstate, int* pbest1, int2* out) {
    static SmemOnce attr;
    if (cudaError_t e = attr(nrw::ladder_fwd_kernel, kSmemFwd)) return e;
    nrw::ladder_fwd_kernel<<<blocks, 32 * nrw::kWarps, kSmemFwd, st>>>(tasks, n_tasks, btasks, pool, sc, scratch, scratch_stride,
                                                                      counter, bvec, ronly, cstate, pbest1, out);
    return cudaGetLastError();
}

}  // namespace nrl
