// nr_launch_gmm_nd.h -- the mixture fits of one or two features (nr_launch_gmm_nd.cu) as the host side (nr_gmm_nd.cu)
// sees them: the problem, start and fit records, the constants both sides use and the launcher.
#pragma once
#include "../../include/nanorepeat_b200.h"
#include <cuda_runtime.h>

namespace nrd {

constexpr int kMaxC = NR_GMM_MAX_COMPONENTS;      // components per mixture
constexpr int kMaxD = 2;                          // features per sample
constexpr int kBigCluster = 8;                    // thread blocks per fit for problems of many samples (portable cluster size)
constexpr int kBigSamples = 16384;                // ... from this many samples on
constexpr double kLog2Pi = 1.8378770664093453;    // log(2 pi)

struct Problem {          // one mixture fit: samples [off, off + count) of data (D values each), n components
    long long off;
    long long region;     // stream id of the random draws
    int count, n;
};

struct Start {            // explicit starting parameters of one problem; m and v are [j * D + d]
    double w[kMaxC], m[kMaxC * kMaxD], v[kMaxC * kMaxD];
};

struct Fit {              // result of one (problem, start); m and v are [j * D + d]
    double lower;
    int iters, converged;
    double w[kMaxC], m[kMaxC * kMaxD], v[kMaxC * kMaxD];
};

}  // namespace nrd

namespace nrl {
// n_starts starts of every problem (p.n_init with the k-means stand-in, 1 with explicit starts), `cluster` thread blocks
// per start (1, or kBigCluster for problems of many samples): fits[problem * n_starts + start].  starts: nullptr, or one
// Start per problem.  n_features: 1 or 2.
cudaError_t launch_gmm_nd_fits(const nr_gmm_params_t& p, int n_features, int n_problems, int n_starts, int cluster, cudaStream_t st,
                               const nrd::Problem* problems, const double* data, const nrd::Start* starts, nrd::Fit* fits);
}  // namespace nrl
