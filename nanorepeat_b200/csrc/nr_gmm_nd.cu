// nr_gmm_nd.cu -- Gaussian-mixture fits of one or two features per sample, many problems per call, on the kernel of
// nr_launch_gmm_nd.cu: what scikit-learn's GaussianMixture(covariance_type='diag').fit does, from explicit starting
// parameters or from the library's k-means stand-in (nanorepeat_b200/mixture.py is the drop-in class on top).
// C ABI: nr_gmm_fit.
#include "nr_internal.h"
#include "nr_launch_gmm_nd.h"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace nrd;

extern "C" int nr_gmm_fit(const nr_gmm_params_t* p, int32_t n_features, int32_t n_problems, const int64_t* offsets,
                          const double* data, const int32_t* n_components, const int64_t* region_id, const double* weights_init,
                          const double* means_init, const double* precisions_init, double* lower, int32_t* iters, uint8_t* converged,
                          double* weights, double* means, double* variances) {
    if (!p || p->max_components < 1 || p->max_components > kMaxC || p->n_init < 1 || p->n_init > 64 || p->max_iter < 1 ||
        !(p->tol >= 0) || !(p->reg_covar >= 0))
        return nri::fail(NR_ERR_ARG, "nr_gmm_fit: bad parameters (1 <= max_components <= %d, 1 <= n_init <= 64, max_iter >= 1, "
                                     "tol >= 0, reg_covar >= 0)", kMaxC);
    if (n_features != 1 && n_features != 2) return nri::fail(NR_ERR_ARG, "nr_gmm_fit: n_features must be 1 or 2, not %d", n_features);
    if (n_problems < 0 || (n_problems > 0 && (!offsets || !data || !n_components || !weights || !means || !variances)))
        return nri::fail(NR_ERR_ARG, "nr_gmm_fit: bad arguments");
    const int given = (weights_init != nullptr) + (means_init != nullptr) + (precisions_init != nullptr);
    if (given != 0 && given != 3) return nri::fail(NR_ERR_ARG, "nr_gmm_fit: give weights_init, means_init and precisions_init together, or none");
    const int D = n_features, C = p->max_components;
    std::vector<Problem> problems(n_problems);
    for (int i = 0; i < n_problems; ++i) {
        const long long cnt = offsets[i + 1] - offsets[i];
        if (offsets[0] != 0 || cnt < 0 || cnt > 0x7fffffff)
            return nri::fail(NR_ERR_ARG, "nr_gmm_fit: offsets must start at 0 and not decrease (at most 2^31 - 1 samples a problem)");
        if (n_components[i] < 1 || n_components[i] > C)
            return nri::fail(NR_ERR_ARG, "nr_gmm_fit: problem %d: n_components = %d, must be in [1, max_components = %d]", i, n_components[i], C);
        if (cnt < n_components[i])
            return nri::fail(NR_ERR_ARG, "nr_gmm_fit: problem %d has %lld samples, fewer than its %d components", i, cnt, n_components[i]);
        problems[i] = {offsets[i], region_id ? region_id[i] : i, (int)cnt, n_components[i]};
    }
    const long long total = n_problems > 0 ? offsets[n_problems] : 0;
    for (long long t = 0; t < total * D; ++t)
        if (!std::isfinite(data[t])) return nri::fail(NR_ERR_ARG, "nr_gmm_fit: sample %lld is not finite", t / D);
    std::vector<Start> starts(given ? n_problems : 0);
    for (int i = 0; i < (int)starts.size(); ++i)
        for (int j = 0; j < n_components[i]; ++j) {
            const double w = weights_init[(size_t)i * C + j];
            if (!(w >= 0 && w <= 1)) return nri::fail(NR_ERR_ARG, "nr_gmm_fit: problem %d: weights_init must lie in [0, 1]", i);
            starts[i].w[j] = w;
            for (int d = 0; d < D; ++d) {
                const double m = means_init[((size_t)i * C + j) * D + d], pr = precisions_init[((size_t)i * C + j) * D + d];
                if (!std::isfinite(m) || !(pr > 0) || !std::isfinite(pr))
                    return nri::fail(NR_ERR_ARG, "nr_gmm_fit: problem %d: means_init must be finite and precisions_init positive", i);
                starts[i].m[j * D + d] = m;
                starts[i].v[j * D + d] = 1.0 / pr;
            }
        }
    int rc = nri::ensure_init();
    if (rc || n_problems == 0) return rc;

    nri::PhaseTrace trace;
    const int n_starts = given ? 1 : p->n_init;          // explicit starts: scikit-learn's n_init starts would all be this one
    const size_t n_fits = (size_t)n_problems * n_starts;
    // problems of few samples first (one thread block per fit), problems of many after them (a cluster of blocks per fit)
    std::vector<int> perm(n_problems);
    for (int i = 0; i < n_problems; ++i) perm[i] = i;
    std::stable_partition(perm.begin(), perm.end(), [&](int i) { return problems[i].count < kBigSamples; });
    int n_small = 0;
    while (n_small < n_problems && problems[perm[n_small]].count < kBigSamples) ++n_small;
    std::vector<Problem> sorted(n_problems);
    std::vector<Start> sorted_starts(starts.size());
    for (int s = 0; s < n_problems; ++s) {
        sorted[s] = problems[perm[s]];
        if (given) sorted_starts[s] = starts[perm[s]];
    }

    nri::Bufs bufs;
    void *d_data = nullptr, *d_prob = nullptr, *d_starts = nullptr, *d_fits = nullptr, *h_fits = nullptr;
    if ((rc = bufs.get(&d_data, sizeof(double) * total * D, false)) || (rc = bufs.get(&d_prob, sizeof(Problem) * n_problems, false)) ||
        (rc = bufs.get(&d_starts, sizeof(Start) * sorted_starts.size(), false)) || (rc = bufs.get(&d_fits, sizeof(Fit) * n_fits, false)) ||
        (rc = bufs.get(&h_fits, sizeof(Fit) * n_fits, true)))
        return rc;
    cudaStream_t st = nri::stream();
    CUDA_TRY(cudaMemcpyAsync(d_data, data, sizeof(double) * total * D, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_prob, sorted.data(), sizeof(Problem) * n_problems, cudaMemcpyHostToDevice, st));
    if (given) CUDA_TRY(cudaMemcpyAsync(d_starts, sorted_starts.data(), sizeof(Start) * n_problems, cudaMemcpyHostToDevice, st));
    const Problem* dp = static_cast<const Problem*>(d_prob);
    const Start* ds = given ? static_cast<const Start*>(d_starts) : nullptr;
    Fit* df = static_cast<Fit*>(d_fits);
    int launches = 0;
    if (n_small > 0) {
        CUDA_TRY(nrl::launch_gmm_nd_fits(*p, D, n_small, n_starts, 1, st, dp, static_cast<const double*>(d_data), ds, df));
        ++launches;
    }
    if (n_problems > n_small) {
        CUDA_TRY(nrl::launch_gmm_nd_fits(*p, D, n_problems - n_small, n_starts, kBigCluster, st, dp + n_small, static_cast<const double*>(d_data),
                                         ds ? ds + n_small : nullptr, df + (size_t)n_small * n_starts));
        ++launches;
    }
    CUDA_TRY(cudaMemcpyAsync(h_fits, d_fits, sizeof(Fit) * n_fits, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    trace.mark("gmm_fit: upload + fits");

    // best start of every problem: the first of the highest lower bounds (scikit-learn's `>`); components in the fit's order
    const Fit* f = static_cast<const Fit*>(h_fits);
    for (int s = 0; s < n_problems; ++s) {
        const int i = perm[s];
        int b = 0;
        for (int k = 1; k < n_starts; ++k)
            if (f[(size_t)s * n_starts + k].lower > f[(size_t)s * n_starts + b].lower) b = k;
        const Fit& best = f[(size_t)s * n_starts + b];
        if (lower) lower[i] = best.lower;
        if (iters) iters[i] = best.iters;
        if (converged) converged[i] = (uint8_t)best.converged;
        for (int j = 0; j < C; ++j) {
            const bool in = j < n_components[i];
            weights[(size_t)i * C + j] = in ? best.w[j] : 0.0;
            for (int d = 0; d < D; ++d) {
                means[((size_t)i * C + j) * D + d] = in ? best.m[j * D + d] : 0.0;
                variances[((size_t)i * C + j) * D + d] = in ? best.v[j * D + d] : 0.0;
            }
        }
    }
    nr_stats_t stats = {};
    stats.n_tasks = (int64_t)n_fits;
    stats.kernel_launches = launches;
    stats.h2d_bytes = (int64_t)(sizeof(double) * total * D + sizeof(Problem) * n_problems + (given ? sizeof(Start) * n_problems : 0));
    stats.d2h_bytes = (int64_t)(sizeof(Fit) * n_fits);
    nri::set_last_stats(stats);
    return NR_OK;
}
