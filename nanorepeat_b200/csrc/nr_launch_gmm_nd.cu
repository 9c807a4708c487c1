// fit_nd_kernel: Gaussian-mixture fits of samples with D = 1 or 2 features and a diagonal covariance, host side in
// nr_gmm_nd.cu.  The same EM as nr_launch_gmm.cu's fit_kernel (scikit-learn's BaseMixture.fit_predict, fp64), with one
// more squared term per feature in the E step and two more sums per feature in the M step.  One 128-thread block per
// (problem, start) -- for problems of many samples a CLUSTER of 8 blocks whose partial sums meet through distributed shared
// memory.  Every iteration is ONE pass over the problem's samples that computes the responsibilities and accumulates the
// 1 + 2D sums per component, followed by a fixed-order reduction (warps, block, cluster ranks: results do not depend on
// scheduling).  Starts: explicit parameters, or the k-means stand-in of oracle/gmm_nd.py (random draws: splitmix64 of
// (seed, region, stream, index), as in the CPU checker).
#include "nr_launch_gmm_nd.h"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;
using namespace nrd;

namespace {

constexpr int kThreads = 128;
constexpr int kLloyd = 10;
constexpr double kEps10 = 10 * 2.220446049250313e-16;

__device__ inline unsigned long long mix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__device__ inline unsigned long long key(unsigned long long seed, long long region, unsigned long long stream, unsigned long long idx) {
    return mix64(mix64(mix64(seed ^ (0xD1B54A32D192ED03ull * (unsigned long long)(region + 1))) + stream) + idx);
}

template <int D> __host__ __device__ constexpr int vals() { return (1 + 2 * D) * kMaxC + 2; }   // the sums of one pass, and the log-likelihood

// Sum of v[0..n) over every thread of the CLUSTER (the thread blocks that share one fit), in a fixed order: warps by
// shuffle, the block's warps in shared memory, the cluster's blocks by rank through distributed shared memory.  Every
// thread of every block may read tot[0..n) afterwards (all blocks hold the same totals, computed in the same order).
template <int D>
__device__ inline void cluster_sum(cg::cluster_group& cluster, double* v, int n, double* red /* [4][vals] */, double* tot /* [vals] */) {
    constexpr int kVals = vals<D>();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = 0; i < n; ++i) {
        double x = v[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) red[warp * kVals + i] = x;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += kThreads) {
        double s = 0;
        for (int w = 0; w < kThreads / 32; ++w) s += red[w * kVals + i];
        red[i] = s;                                 // (row 0 of warp 0 is overwritten by its own column's total)
    }
    const unsigned nb = cluster.num_blocks();
    if (nb == 1) {
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += kThreads) tot[i] = red[i];
        __syncthreads();
        return;
    }
    cluster.sync();                                 // every block's partial sums are in its red[0..n)
    for (int i = threadIdx.x; i < n; i += kThreads) {
        double s = 0;
        for (unsigned r = 0; r < nb; ++r) s += cluster.map_shared_rank(red, r)[i];
        tot[i] = s;
    }
    cluster.sync();                                 // nobody overwrites red while a neighbour still reads it
}

// One fit = one cluster of thread blocks: cluster `blockIdx.x / cluster size` is (problem, start).  Every block walks its
// share of the samples, the sums meet in cluster_sum, and every block then updates the same parameters redundantly.
// Sums of a pass: acc[j] = sum r, acc[n + j*D + d] = sum r x_d, acc[n + n*D + j*D + d] = sum r x_d^2, acc[(1 + 2D) n] =
// sum of the log-likelihoods -- at D = 1 the layout and the arithmetic of fit_kernel.
template <int D>
__global__ void __launch_bounds__(kThreads)
fit_nd_kernel(const Problem* __restrict__ problems, const double* __restrict__ data, const Start* __restrict__ starts, int n_starts,
              int max_iter, double tol, double reg_covar, unsigned long long seed, Fit* __restrict__ fits) {
    constexpr int kVals = vals<D>();
    cg::cluster_group cluster = cg::this_cluster();
    const int nb = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int fit = (int)(blockIdx.x / nb);
    __shared__ double red[(kThreads / 32) * kVals];
    __shared__ double tot[kVals];
    __shared__ double sw[kMaxC], sm[kMaxC * D], sv[kMaxC * D], spc[kMaxC * D], sc0[kMaxC];
    const Problem pb = problems[fit / n_starts];
    const int init = fit % n_starts, n = pb.n, N = pb.count;
    const double* x = data + pb.off * D;
    const int first = rank * kThreads + (int)threadIdx.x, stride = nb * kThreads;      // this thread's samples
    double acc[kVals];

    if (starts) {                                   // ---- explicit start (weights_init / means_init / precisions_init)
        const Start& s = starts[fit / n_starts];
        if (threadIdx.x < n) {
            const int j = threadIdx.x;
            sw[j] = s.w[j];
            for (int d = 0; d < D; ++d) { sm[j * D + d] = s.m[j * D + d]; sv[j * D + d] = s.v[j * D + d]; }
        }
        __syncthreads();
    } else {
        // ---- start: means (init 0: evenly along the bounding box's diagonal; else hashed sample rows), kLloyd rounds of
        // k-means on the squared Euclidean distance (|x - m| at D = 1: the same order), the one-hot M step
        if (init == 0) {
            double lo[D], hi[D];
            for (int d = 0; d < D; ++d) { lo[d] = 1e300; hi[d] = -1e300; }
            for (int i = first; i < N; i += stride)
                for (int d = 0; d < D; ++d) { lo[d] = fmin(lo[d], x[(long long)i * D + d]); hi[d] = fmax(hi[d], x[(long long)i * D + d]); }
            for (int d = 0; d < D; ++d) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    lo[d] = fmin(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
                    hi[d] = fmax(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
                }
                if ((threadIdx.x & 31) == 0) { red[(threadIdx.x >> 5) * 2 * D + d] = lo[d]; red[(threadIdx.x >> 5) * 2 * D + D + d] = hi[d]; }
            }
            __syncthreads();
            if (threadIdx.x == 0)
                for (int d = 0; d < D; ++d) {
                    red[8 * D + d] = fmin(fmin(red[d], red[2 * D + d]), fmin(red[4 * D + d], red[6 * D + d]));
                    red[9 * D + d] = fmax(fmax(red[D + d], red[3 * D + d]), fmax(red[5 * D + d], red[7 * D + d]));
                }
            if (nb > 1) cluster.sync(); else __syncthreads();
            for (int d = 0; d < D; ++d) { lo[d] = 1e300; hi[d] = -1e300; }
            for (int r = 0; r < nb; ++r) {
                const double* rr = nb > 1 ? cluster.map_shared_rank(red, r) : red;
                for (int d = 0; d < D; ++d) { lo[d] = fmin(lo[d], rr[8 * D + d]); hi[d] = fmax(hi[d], rr[9 * D + d]); }
            }
            if (nb > 1) cluster.sync(); else __syncthreads();
            if (threadIdx.x < n)
                for (int d = 0; d < D; ++d) sm[threadIdx.x * D + d] = lo[d] + (threadIdx.x + 0.5) / n * (hi[d] - lo[d]);
        } else if (threadIdx.x < n) {
            const long long row = (long long)(key(seed, pb.region, 1000 + 32 * n + init, threadIdx.x) % (unsigned long long)N);
            for (int d = 0; d < D; ++d) sm[threadIdx.x * D + d] = x[row * D + d];
        }
        __syncthreads();
        for (int round = 0; round <= kLloyd; ++round) {
            // labels by the nearest mean (lowest index on ties); the last round turns them into the first M step
            for (int j = 0; j < (1 + 2 * D) * n; ++j) acc[j] = 0;
            for (int i = first; i < N; i += stride) {
                double xi[D];
                for (int d = 0; d < D; ++d) xi[d] = x[(long long)i * D + d];
                int lab = 0;
                double bd = 0;
                for (int j = 0; j < n; ++j) {
                    double dist;
                    if (D == 1) {
                        dist = fabs(xi[0] - sm[j]);
                    } else {
                        dist = 0;
                        for (int d = 0; d < D; ++d) { const double e = xi[d] - sm[j * D + d]; dist += e * e; }
                    }
                    if (j == 0 || dist < bd) { bd = dist; lab = j; }
                }
                acc[lab] += 1.0;
                for (int d = 0; d < D; ++d) { acc[n + lab * D + d] += xi[d]; acc[n + n * D + lab * D + d] += xi[d] * xi[d]; }
            }
            cluster_sum<D>(cluster, acc, (1 + 2 * D) * n, red, tot);
            if (threadIdx.x < n) {
                const int j = threadIdx.x;
                if (round < kLloyd) {
                    if (tot[j] > 0)
                        for (int d = 0; d < D; ++d) sm[j * D + d] = tot[n + j * D + d] / tot[j];
                } else {      // sklearn _estimate_gaussian_parameters on one-hot responsibilities
                    const double nk = tot[j] + kEps10;
                    sw[j] = nk / N;
                    for (int d = 0; d < D; ++d) {
                        const double mean = tot[n + j * D + d] / nk;
                        sm[j * D + d] = mean; sv[j * D + d] = tot[n + n * D + j * D + d] / nk - mean * mean + reg_covar;
                    }
                }
            }
            __syncthreads();
        }
    }

    // ---- EM (BaseMixture.fit_predict: E step, M step, |change of the mean log-likelihood| < tol)
    double lower = -INFINITY;
    int iters = 0, converged = 0;
    for (int it = 1; it <= max_iter; ++it) {
        if (threadIdx.x < n) {
            const int j = threadIdx.x;
            double c = 0;
            for (int d = 0; d < D; ++d) {
                const double pc = 1.0 / sqrt(sv[j * D + d]);
                spc[j * D + d] = pc;
                c += log(pc);
            }
            sc0[j] = c + log(sw[j]) - 0.5 * D * kLog2Pi;
        }
        __syncthreads();
        for (int j = 0; j < (1 + 2 * D) * n + 1; ++j) acc[j] = 0;
        for (int i = first; i < N; i += stride) {
            double xi[D];
            for (int d = 0; d < D; ++d) xi[d] = x[(long long)i * D + d];
            double lp[kMaxC];
            double top = -INFINITY;
            for (int j = 0; j < n; ++j) {
                double q = 0;
                for (int d = 0; d < D; ++d) { const double e = (xi[d] - sm[j * D + d]) * spc[j * D + d]; q += e * e; }
                lp[j] = sc0[j] - 0.5 * q;
                top = fmax(top, lp[j]);
            }
            double s = 0;
            for (int j = 0; j < n; ++j) s += exp(lp[j] - top);
            const double norm = top + log(s);
            for (int j = 0; j < n; ++j) {
                const double r = exp(lp[j] - norm);
                acc[j] += r;
                for (int d = 0; d < D; ++d) { acc[n + j * D + d] += r * xi[d]; acc[n + n * D + j * D + d] += r * xi[d] * xi[d]; }
            }
            acc[(1 + 2 * D) * n] += norm;
        }
        cluster_sum<D>(cluster, acc, (1 + 2 * D) * n + 1, red, tot);
        const double prev = lower;
        lower = tot[(1 + 2 * D) * n] / N;
        __syncthreads();
        if (threadIdx.x < n) {
            const int j = threadIdx.x;
            const double nk = tot[j] + kEps10;
            sw[j] = nk / N;
            for (int d = 0; d < D; ++d) {
                const double mean = tot[n + j * D + d] / nk;
                sm[j * D + d] = mean; sv[j * D + d] = tot[n + n * D + j * D + d] / nk - mean * mean + reg_covar;
            }
        }
        __syncthreads();
        iters = it;
        if (fabs(lower - prev) < tol) { converged = 1; break; }        // (the same number in every block: all leave together)
    }
    if (rank == 0) {
        Fit& f = fits[fit];
        if (threadIdx.x == 0) { f.lower = lower; f.iters = iters; f.converged = converged; }
        if (threadIdx.x < n) {
            const int j = threadIdx.x;
            f.w[j] = sw[j];
            for (int d = 0; d < D; ++d) { f.m[j * D + d] = sm[j * D + d]; f.v[j * D + d] = sv[j * D + d]; }
        }
    }
}

template <int D>
cudaError_t launch(const nr_gmm_params_t& p, int n_problems, int n_starts, int cluster, cudaStream_t st, const Problem* problems,
                   const double* data, const Start* starts, Fit* fits) {
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = (unsigned)cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((size_t)n_problems * n_starts * cluster));
    cfg.blockDim = dim3(kThreads);
    cfg.stream = st; cfg.attrs = &attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, fit_nd_kernel<D>, problems, data, starts, n_starts, (int)p.max_iter, (double)p.tol,
                              (double)p.reg_covar, (unsigned long long)p.seed, fits);
}

}  // namespace

namespace nrl {

cudaError_t launch_gmm_nd_fits(const nr_gmm_params_t& p, int n_features, int n_problems, int n_starts, int cluster, cudaStream_t st,
                               const Problem* problems, const double* data, const Start* starts, Fit* fits) {
    if (n_problems == 0) return cudaSuccess;
    if (n_features == 1) return launch<1>(p, n_problems, n_starts, cluster, st, problems, data, starts, fits);
    return launch<2>(p, n_problems, n_starts, cluster, st, problems, data, starts, fits);
}

}  // namespace nrl
