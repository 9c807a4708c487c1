// bootstrap_kernel, fit_kernel: the batched 1-D Gaussian-mixture phasing, host side in nr_gmm.cu.  One 128-thread block
// per (region, start) runs the whole EM of that start in fp64 -- for regions of many samples (amplicon data: thousands of
// reads) a CLUSTER of 8 blocks whose partial sums meet through distributed shared memory: every iteration is ONE pass
// over the region's bootstrapped sizes that computes the responsibilities (E step) and accumulates the M step's three
// sums per component, followed by a fixed-order reduction (warps, block, cluster ranks: results do not depend on
// scheduling).  Random draws: splitmix64 of (seed, region, stream, index), as in the CPU checker.
#include "nr_launch_gmm.h"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;
using namespace nrg;

namespace {

constexpr int kThreads = 128;
constexpr int kLloyd = 10;
constexpr double kEps10 = 10 * 2.220446049250313e-16;

__host__ __device__ inline unsigned long long mix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__host__ __device__ inline unsigned long long key(unsigned long long seed, long long region, unsigned long long stream, unsigned long long idx) {
    return mix64(mix64(mix64(seed ^ (0xD1B54A32D192ED03ull * (unsigned long long)(region + 1))) + stream) + idx);
}
__device__ inline double uniform01(unsigned long long h) { return (double)((h >> 11) + 1) * (1.0 / 9007199254740992.0); }

// sample rep * n + i of a region = x[i] + N(0, error_rate * (10 + x[i]))       (split_alleles.py:82-88)
__global__ void bootstrap_kernel(const double* __restrict__ sizes, const long long* __restrict__ off, int n_regions, long long region_base,
                                 double error_rate, unsigned long long seed, double* __restrict__ out) {
    for (int g = blockIdx.x; g < n_regions; g += gridDim.x) {
        const long long o = off[g], n = off[g + 1] - o;
        for (long long t = threadIdx.x; t < n * kBootstrap; t += blockDim.x) {
            const double x = sizes[o + t % n];
            const double u1 = uniform01(key(seed, region_base + g, 1, (unsigned long long)t));
            const double u2 = uniform01(key(seed, region_base + g, 2, (unsigned long long)t));
            const double z = sqrt(-2.0 * log(u1)) * cos(2.0 * 3.14159265358979323846 * u2);
            out[o * kBootstrap + t] = x + error_rate * (10.0 + x) * z;
        }
    }
}

constexpr int kVals = 3 * kMaxC + 2;

// Sum of v[0..n) over every thread of the CLUSTER (the thread blocks that share one fit), in a fixed order: warps by
// shuffle, the block's warps in shared memory, the cluster's blocks by rank through distributed shared memory.  Every
// thread of every block may read tot[0..n) afterwards (all blocks hold the same totals, computed in the same order).
__device__ inline void cluster_sum(cg::cluster_group& cluster, double* v, int n, double* red /* [4][kVals] */, double* tot /* [kVals] */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = 0; i < n; ++i) {
        double x = v[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) red[warp * kVals + i] = x;
    }
    __syncthreads();
    if (threadIdx.x < n) {
        double s = 0;
        for (int w = 0; w < kThreads / 32; ++w) s += red[w * kVals + threadIdx.x];
        red[threadIdx.x] = s;                       // (row 0 of warp 0 is overwritten by its own column's total)
    }
    const unsigned nb = cluster.num_blocks();
    if (nb == 1) {
        __syncthreads();
        if (threadIdx.x < n) tot[threadIdx.x] = red[threadIdx.x];
        __syncthreads();
        return;
    }
    cluster.sync();                                 // every block's partial sums are in its red[0..n)
    if (threadIdx.x < n) {
        double s = 0;
        for (unsigned r = 0; r < nb; ++r) s += cluster.map_shared_rank(red, r)[threadIdx.x];
        tot[threadIdx.x] = s;
    }
    cluster.sync();                                 // nobody overwrites red while a neighbour still reads it
}

// One fit = one cluster of thread blocks (one block for small regions, kBigCluster for regions of many samples):
// cluster `blockIdx.x / cluster size` is (problem, start).  Every block of the cluster walks its share of the samples,
// the sums meet in cluster_sum, and every block then updates the same parameters redundantly (no broadcast).
__global__ void __launch_bounds__(kThreads)
fit_kernel(const Problem* __restrict__ problems, const double* __restrict__ data, int n_init, int max_iter, double tol, double reg_covar,
           unsigned long long seed, Fit* __restrict__ fits) {
    cg::cluster_group cluster = cg::this_cluster();
    const int nb = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int fit = (int)(blockIdx.x / nb);
    __shared__ double red[(kThreads / 32) * kVals];
    __shared__ double tot[kVals];
    __shared__ double sw[kMaxC], sm[kMaxC], sv[kMaxC], spc[kMaxC], sc0[kMaxC];
    const Problem pb = problems[fit / n_init];
    const int init = fit % n_init, n = pb.n, N = pb.count;
    const double* x = data + pb.off;
    const int first = rank * kThreads + (int)threadIdx.x, stride = nb * kThreads;      // this thread's samples
    double acc[kVals];

    // ---- start: means (init 0: evenly over [min, max]; else hashed sample positions), kLloyd rounds of 1-D k-means
    if (init == 0) {
        double lo = 1e300, hi = -1e300;
        for (int i = first; i < N; i += stride) { lo = fmin(lo, x[i]); hi = fmax(hi, x[i]); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o)); }
        if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = lo; red[4 + (threadIdx.x >> 5)] = hi; }
        __syncthreads();
        if (threadIdx.x == 0) {
            red[8] = fmin(fmin(red[0], red[1]), fmin(red[2], red[3]));
            red[9] = fmax(fmax(red[4], red[5]), fmax(red[6], red[7]));
        }
        if (nb > 1) cluster.sync(); else __syncthreads();
        lo = 1e300; hi = -1e300;
        for (int r = 0; r < nb; ++r) {
            const double* rr = nb > 1 ? cluster.map_shared_rank(red, r) : red;
            lo = fmin(lo, rr[8]); hi = fmax(hi, rr[9]);
        }
        if (nb > 1) cluster.sync(); else __syncthreads();
        if (threadIdx.x < n) sm[threadIdx.x] = lo + (threadIdx.x + 0.5) / n * (hi - lo);
    } else if (threadIdx.x < n) {
        sm[threadIdx.x] = x[key(seed, pb.region, 1000 + 32 * n + init, threadIdx.x) % (unsigned long long)N];
    }
    __syncthreads();
    for (int round = 0; round <= kLloyd; ++round) {
        // labels by the nearest mean (lowest index on ties); the last round turns them into the first M step
        for (int j = 0; j < 3 * n; ++j) acc[j] = 0;
        for (int i = first; i < N; i += stride) {
            const double xi = x[i];
            int lab = 0;
            double bd = fabs(xi - sm[0]);
            for (int j = 1; j < n; ++j) { const double d = fabs(xi - sm[j]); if (d < bd) { bd = d; lab = j; } }
            acc[lab] += 1.0; acc[n + lab] += xi; acc[2 * n + lab] += xi * xi;
        }
        cluster_sum(cluster, acc, 3 * n, red, tot);
        if (threadIdx.x < n) {
            const int j = threadIdx.x;
            if (round < kLloyd) {
                if (tot[j] > 0) sm[j] = tot[n + j] / tot[j];
            } else {          // sklearn _estimate_gaussian_parameters on one-hot responsibilities
                const double nk = tot[j] + kEps10;
                const double mean = tot[n + j] / nk;
                sw[j] = nk / N; sm[j] = mean; sv[j] = tot[2 * n + j] / nk - mean * mean + reg_covar;
            }
        }
        __syncthreads();
    }

    // ---- EM (BaseMixture.fit_predict: E step, M step, |change of the mean log-likelihood| < tol)
    double lower = -INFINITY;
    int iters = 0, converged = 0;
    for (int it = 1; it <= max_iter; ++it) {
        if (threadIdx.x < n) {
            const int j = threadIdx.x;
            const double pc = 1.0 / sqrt(sv[j]);
            spc[j] = pc;
            sc0[j] = log(pc) + log(sw[j]) - 0.5 * kLog2Pi;
        }
        __syncthreads();
        for (int j = 0; j < 3 * n + 1; ++j) acc[j] = 0;
        for (int i = first; i < N; i += stride) {
            const double xi = x[i];
            double lp[kMaxC];
            double top = -INFINITY;
            for (int j = 0; j < n; ++j) {
                const double d = (xi - sm[j]) * spc[j];
                lp[j] = sc0[j] - 0.5 * d * d;
                top = fmax(top, lp[j]);
            }
            double s = 0;
            for (int j = 0; j < n; ++j) s += exp(lp[j] - top);
            const double norm = top + log(s);
            for (int j = 0; j < n; ++j) {
                const double r = exp(lp[j] - norm);
                acc[j] += r; acc[n + j] += r * xi; acc[2 * n + j] += r * xi * xi;
            }
            acc[3 * n] += norm;
        }
        cluster_sum(cluster, acc, 3 * n + 1, red, tot);
        const double prev = lower;
        lower = tot[3 * n] / N;
        __syncthreads();
        if (threadIdx.x < n) {
            const int j = threadIdx.x;
            const double nk = tot[j] + kEps10;
            const double mean = tot[n + j] / nk;
            sw[j] = nk / N; sm[j] = mean; sv[j] = tot[2 * n + j] / nk - mean * mean + reg_covar;
        }
        __syncthreads();
        iters = it;
        if (fabs(lower - prev) < tol) { converged = 1; break; }        // (the same number in every block: all leave together)
    }
    if (rank == 0) {
        Fit& f = fits[fit];
        if (threadIdx.x == 0) { f.lower = lower; f.iters = iters; f.converged = converged; }
        if (threadIdx.x < n) { f.w[threadIdx.x] = sw[threadIdx.x]; f.m[threadIdx.x] = sm[threadIdx.x]; f.v[threadIdx.x] = sv[threadIdx.x]; }
    }
}

}  // namespace

namespace nrl {

cudaError_t launch_gmm_bootstrap(const nr_gmm_params_t& p, int blocks, cudaStream_t st, const double* sizes, const long long* off,
                                 int n_regions, long long region_base, double* out) {
    bootstrap_kernel<<<blocks, 256, 0, st>>>(sizes, off, n_regions, region_base, p.error_rate, p.seed, out);
    return cudaGetLastError();
}

cudaError_t launch_gmm_fits(const nr_gmm_params_t& p, int n_problems, int cluster, cudaStream_t st, const Problem* problems,
                            const double* data, Fit* fits) {
    if (n_problems == 0) return cudaSuccess;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = (unsigned)cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((size_t)n_problems * p.n_init * cluster));
    cfg.blockDim = dim3(kThreads);
    cfg.stream = st; cfg.attrs = &attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, fit_kernel, problems, data, (int)p.n_init, (int)p.max_iter, (double)p.tol, (double)p.reg_covar,
                              (unsigned long long)p.seed, fits);
}

}  // namespace nrl
