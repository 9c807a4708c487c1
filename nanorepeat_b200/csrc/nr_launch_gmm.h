// nr_launch_gmm.h -- the phasing's kernels (nr_launch_gmm.cu) as the host side (nr_gmm.cu) sees them: the problem and
// fit records, the constants both sides use and one launcher per kernel, each returning the launch's cudaError_t.
#pragma once
#include "../../include/nanorepeat_b200.h"
#include <cuda_runtime.h>

namespace nrg {

constexpr int kMaxC = NR_GMM_MAX_COMPONENTS;      // components per mixture
constexpr int kBootstrap = 100;                   // split_alleles.py:83
constexpr int kBigCluster = 8;                    // thread blocks per fit for regions of many samples (portable cluster size)
constexpr int kBigSamples = 16384;                // ... from this many bootstrapped samples on
constexpr double kLog2Pi = 1.8378770664093453;    // log(2 pi)

struct Problem {          // one mixture fit: data[off .. off + count), n components
    long long off;
    long long region;     // stream id of the random draws
    int count, n;
};

struct Fit {              // result of one (problem, start)
    double lower;
    int iters, converged;
    double w[kMaxC], m[kMaxC], v[kMaxC];
};

}  // namespace nrg

namespace nrl {
// sample rep * n + i of region g = sizes[off[g] + i] + noise, out[off[g] * kBootstrap + rep * n + i]; 256 threads a block
cudaError_t launch_gmm_bootstrap(const nr_gmm_params_t& p, int blocks, cudaStream_t st, const double* sizes, const long long* off,
                                 int n_regions, long long region_base, double* out);
// p.n_init starts of every problem, `cluster` thread blocks per start (1, or kBigCluster for problems of many samples):
// fits[problem * n_init + start]
cudaError_t launch_gmm_fits(const nr_gmm_params_t& p, int n_problems, int cluster, cudaStream_t st, const nrg::Problem* problems,
                            const double* data, nrg::Fit* fits);
}  // namespace nrl
