// nr_gmm.cu -- batched 1-D Gaussian-mixture phasing (SURVEY.md 8(f) row f3): what the reference does per region after
// round 3 (nanoRepeat_bam.py:515-575, split_alleles.py:82-200) -- 3-sigma trim, 100x bootstrap with Gaussian noise
// sd = error_rate * (10 + size), GaussianMixture(n, 'diag', n_init = 10) for n = 2, 3, ... until two components'
// [isf(1 - o), isf(o)] intervals overlap -- for many regions at once, on the kernels of nr_launch_gmm.cu.  The stopping
// rule, the regularisation and the choice among the starts are scikit-learn's (BaseMixture.fit_predict); the random
// draws are not: the reference uses unseeded generators (random.gauss, sklearn's k-means), this library a counter-based
// one that the CPU checker shares -- a phased region is reproducible, and independent of how regions are batched.
// C ABI: nr_gmm_bootstrap, nr_gmm1d_fit, nr_phase_1d.
#include "nr_internal.h"
#include "nr_launch_gmm.h"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace nrg;

namespace {

int check_params(const nr_gmm_params_t* p) {
    if (!p || p->max_components < 1 || p->max_components > kMaxC || p->n_init < 1 || p->n_init > 64 || p->max_iter < 1 ||
        !(p->tol > 0) || !(p->reg_covar >= 0) || !(p->error_rate >= 0) || !(p->max_mutual_overlap > 0 && p->max_mutual_overlap < 1))
        return nri::fail(NR_ERR_ARG, "nr_gmm: bad parameters (1 <= max_components <= NR_GMM_MAX_COMPONENTS, 1 <= n_init <= 64, 0 < overlap < 1)");
    return NR_OK;
}

// scipy.stats.norm.isf(o) of the standard normal, by Newton on erfc
double std_isf(double o) {
    double z = 0;
    for (int i = 0; i < 60; ++i) z += (0.5 * erfc(z / sqrt(2.0)) - o) / (exp(-0.5 * z * z) / sqrt(2.0 * 3.14159265358979323846));
    return z;
}

// split_alleles.py:176-195
bool any_overlap(const Fit& f, int n, double z) {
    for (int i = 0; i < n; ++i)
        for (int j = i + 1; j < n; ++j) {
            const double si = std::max(1.0, sqrt(f.v[i])), sj = std::max(1.0, sqrt(f.v[j]));
            const double lo = std::max(f.m[i] - z * si, f.m[j] - z * sj), hi = std::min(f.m[i] + z * si, f.m[j] + z * sj);
            if (lo - hi <= 0) return true;
        }
    return false;
}

// Best start of every problem (first of the highest lower bounds, as sklearn's `>`).  d_data: the problems' samples.
int run_fits(const nr_gmm_params_t* p, const std::vector<Problem>& problems, const double* d_data, std::vector<Fit>& best) {
    const int np = (int)problems.size();
    best.resize(np);
    if (np == 0) return NR_OK;
    const size_t n_fits = (size_t)np * p->n_init;
    nri::Bufs bufs;
    void *d_prob = nullptr, *d_fits = nullptr, *h_fits = nullptr;
    int rc;
    if ((rc = bufs.get(&d_prob, sizeof(Problem) * np, false)) || (rc = bufs.get(&d_fits, sizeof(Fit) * n_fits, false)) ||
        (rc = bufs.get(&h_fits, sizeof(Fit) * n_fits, true)))
        return rc;
    cudaStream_t st = nri::stream();
    // regions of few samples first (one thread block per fit), regions of many after them (a cluster of blocks per fit)
    std::vector<int> perm(np);
    for (int i = 0; i < np; ++i) perm[i] = i;
    std::stable_partition(perm.begin(), perm.end(), [&](int i) { return problems[i].count < kBigSamples; });
    int n_small = 0;
    while (n_small < np && problems[perm[n_small]].count < kBigSamples) ++n_small;
    std::vector<Problem> sorted(np);
    for (int i = 0; i < np; ++i) sorted[i] = problems[perm[i]];
    CUDA_TRY(cudaMemcpyAsync(d_prob, sorted.data(), sizeof(Problem) * np, cudaMemcpyHostToDevice, st));
    CUDA_TRY(nrl::launch_gmm_fits(*p, n_small, 1, st, static_cast<const Problem*>(d_prob), d_data, static_cast<Fit*>(d_fits)));
    CUDA_TRY(nrl::launch_gmm_fits(*p, np - n_small, kBigCluster, st, static_cast<const Problem*>(d_prob) + n_small, d_data,
                                  static_cast<Fit*>(d_fits) + (size_t)n_small * p->n_init));
    CUDA_TRY(cudaMemcpyAsync(h_fits, d_fits, sizeof(Fit) * n_fits, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const Fit* f = static_cast<const Fit*>(h_fits);
    for (int s = 0; s < np; ++s) {
        const int i = perm[s];
        int b = 0;
        for (int k = 1; k < p->n_init; ++k)
            if (f[(size_t)s * p->n_init + k].lower > f[(size_t)s * p->n_init + b].lower) b = k;
        best[i] = f[(size_t)s * p->n_init + b];
        // components in ascending order of their means: which start won a near tie must not show in the result
        const int n = problems[i].n;
        int order[kMaxC];
        for (int j = 0; j < n; ++j) order[j] = j;
        const Fit& src = f[(size_t)s * p->n_init + b];
        std::stable_sort(order, order + n, [&](int a, int c) { return src.m[a] < src.m[c]; });
        for (int j = 0; j < n; ++j) { best[i].w[j] = src.w[order[j]]; best[i].m[j] = src.m[order[j]]; best[i].v[j] = src.v[order[j]]; }
    }
    return NR_OK;
}

int upload_and_bootstrap(const nr_gmm_params_t* p, int n_regions, const std::vector<long long>& off, const double* sizes, long long region_base,
                         nri::Bufs& bufs, double** d_sim) {
    const long long total = off[n_regions];
    void *d_sizes = nullptr, *d_off = nullptr, *sim = nullptr;
    int rc;
    if ((rc = bufs.get(&d_sizes, sizeof(double) * total, false)) || (rc = bufs.get(&d_off, sizeof(long long) * (n_regions + 1), false)) ||
        (rc = bufs.get(&sim, sizeof(double) * total * kBootstrap, false)))
        return rc;
    cudaStream_t st = nri::stream();
    CUDA_TRY(cudaMemcpyAsync(d_sizes, sizes, sizeof(double) * total, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_off, off.data(), sizeof(long long) * (n_regions + 1), cudaMemcpyHostToDevice, st));
    const int blocks = std::max(1, std::min(n_regions, 8 * nri::sm_count()));
    CUDA_TRY(nrl::launch_gmm_bootstrap(*p, blocks, st, static_cast<const double*>(d_sizes), static_cast<const long long*>(d_off), n_regions,
                                       region_base, static_cast<double*>(sim)));
    *d_sim = static_cast<double*>(sim);
    return NR_OK;
}

}  // namespace

extern "C" int nr_gmm_bootstrap(const nr_gmm_params_t* p, int32_t n_regions, const int64_t* offsets, const double* sizes,
                                int64_t region_id_base, double* out) {
    if (check_params(p)) return nri::last_code();
    if (n_regions < 0 || (n_regions > 0 && (!offsets || !sizes || !out))) return nri::fail(NR_ERR_ARG, "nr_gmm_bootstrap: bad arguments");
    int rc = nri::ensure_init();
    if (rc || n_regions == 0) return rc;
    std::vector<long long> off(offsets, offsets + n_regions + 1);
    for (int g = 0; g < n_regions; ++g)
        if (off[g + 1] < off[g] || off[0] != 0) return nri::fail(NR_ERR_ARG, "nr_gmm_bootstrap: offsets must start at 0 and not decrease");
    if (off[n_regions] == 0) return NR_OK;
    nri::Bufs bufs;
    double* d_sim = nullptr;
    if ((rc = upload_and_bootstrap(p, n_regions, off, sizes, region_id_base, bufs, &d_sim))) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, d_sim, sizeof(double) * off[n_regions] * kBootstrap, cudaMemcpyDeviceToHost, nri::stream()));
    CUDA_TRY(cudaStreamSynchronize(nri::stream()));
    return NR_OK;
}

extern "C" int nr_gmm1d_fit(const nr_gmm_params_t* p, int32_t n_problems, const int64_t* offsets, const double* data,
                            const int32_t* n_components, const int64_t* region_id, double* lower, int32_t* iters,
                            double* weights, double* means, double* variances) {
    if (check_params(p)) return nri::last_code();
    if (n_problems < 0 || (n_problems > 0 && (!offsets || !data || !n_components || !weights || !means || !variances)))
        return nri::fail(NR_ERR_ARG, "nr_gmm1d_fit: bad arguments");
    int rc = nri::ensure_init();
    if (rc || n_problems == 0) return rc;
    std::vector<Problem> problems(n_problems);
    for (int i = 0; i < n_problems; ++i) {
        const long long cnt = offsets[i + 1] - offsets[i];
        if (offsets[0] != 0 || cnt < 1 || cnt > 0x7fffffff || n_components[i] < 1 || n_components[i] > p->max_components)
            return nri::fail(NR_ERR_ARG, "nr_gmm1d_fit: every problem needs >= 1 sample and 1 <= n_components <= max_components");
        problems[i] = {offsets[i], region_id ? region_id[i] : i, (int)cnt, n_components[i]};
    }
    nri::Bufs bufs;
    void* d_data = nullptr;
    if ((rc = bufs.get(&d_data, sizeof(double) * offsets[n_problems], false))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_data, data, sizeof(double) * offsets[n_problems], cudaMemcpyHostToDevice, nri::stream()));
    std::vector<Fit> best;
    if ((rc = run_fits(p, problems, static_cast<const double*>(d_data), best))) return rc;
    for (int i = 0; i < n_problems; ++i) {
        if (lower) lower[i] = best[i].lower;
        if (iters) iters[i] = best[i].iters;
        for (int j = 0; j < p->max_components; ++j) {
            const bool in = j < n_components[i];
            weights[(size_t)i * p->max_components + j] = in ? best[i].w[j] : 0.0;
            means[(size_t)i * p->max_components + j] = in ? best[i].m[j] : 0.0;
            variances[(size_t)i * p->max_components + j] = in ? best[i].v[j] : 0.0;
        }
    }
    return NR_OK;
}

extern "C" int nr_phase_1d(const nr_gmm_params_t* p, int32_t n_regions, const int64_t* offsets, const double* sizes,
                           int64_t region_id_base, int32_t* n_components, double* weights, double* means, double* variances,
                           int32_t* label, double* proba) {
    if (check_params(p)) return nri::last_code();
    if (n_regions < 0 || (n_regions > 0 && (!offsets || !n_components || !weights || !means || !variances)))
        return nri::fail(NR_ERR_ARG, "nr_phase_1d: bad arguments");
    int rc = nri::ensure_init();
    if (rc || n_regions == 0) return rc;
    if (offsets[0] != 0) return nri::fail(NR_ERR_ARG, "nr_phase_1d: offsets must start at 0");
    const long long total = offsets[n_regions];
    if (total > 0 && (!sizes || !label || !proba)) return nri::fail(NR_ERR_ARG, "nr_phase_1d: bad arguments");
    const int C = p->max_components;
    for (long long i = 0; i < total; ++i) { label[i] = -1; proba[i] = 0.0; }
    for (size_t i = 0; i < (size_t)n_regions * C; ++i) weights[i] = means[i] = variances[i] = 0.0;

    // ---- 3-sigma trim per region (split_alleles.py:98-113, :141-154); regions with fewer than two sizes are not phased
    // (nanoRepeat_bam.py:533-539)
    std::vector<long long> toff(n_regions + 1, 0);
    std::vector<double> kept;
    std::vector<long long> kept_src;
    kept.reserve((size_t)total);
    kept_src.reserve((size_t)total);
    for (int g = 0; g < n_regions; ++g) {
        const long long a = offsets[g], b = offsets[g + 1];
        if (b < a) return nri::fail(NR_ERR_ARG, "nr_phase_1d: offsets must not decrease");
        n_components[g] = 0;
        if (b - a >= 2) {
            if ((b - a) * (long long)kBootstrap > 0x7fffffff) return nri::fail(NR_ERR_TOO_LARGE, "nr_phase_1d: more than 21 million sizes in one region");
            double s = 0;
            for (long long i = a; i < b; ++i) s += sizes[i];
            const double mean = s / (double)(b - a);
            double q = 0;
            for (long long i = a; i < b; ++i) q += (sizes[i] - mean) * (sizes[i] - mean);
            const double sd = sqrt(q / (double)(b - a));
            const double lo = std::max(mean - 3 * sd, 0.0), hi = mean + 3 * sd;
            for (long long i = a; i < b; ++i)
                if (!(sizes[i] < lo || sizes[i] > hi)) { kept.push_back(sizes[i]); kept_src.push_back(i); }
        }
        toff[g + 1] = (long long)kept.size();
    }
    if (kept.empty()) return NR_OK;

    nri::Bufs bufs;
    double* d_sim = nullptr;
    if ((rc = upload_and_bootstrap(p, n_regions, toff, kept.data(), region_id_base, bufs, &d_sim))) return rc;

    // ---- auto-GMM in waves (split_alleles.py:171-200): wave n fits n components for every region still growing
    const double z = std_isf(p->max_mutual_overlap);
    std::vector<Fit> chosen(n_regions);
    std::vector<int> active;
    std::vector<Problem> problems;
    for (int g = 0; g < n_regions; ++g)
        if (toff[g + 1] > toff[g]) { active.push_back(g); problems.push_back({toff[g] * kBootstrap, region_id_base + g, (int)((toff[g + 1] - toff[g]) * kBootstrap), 1}); }
    {   // one component: the sample mean and variance (one start is enough)
        nr_gmm_params_t one = *p;
        one.n_init = 1;
        std::vector<Fit> best;
        if ((rc = run_fits(&one, problems, d_sim, best))) return rc;
        for (size_t i = 0; i < active.size(); ++i) { chosen[active[i]] = best[i]; n_components[active[i]] = 1; }
    }
    for (int n = 2; n <= C && !active.empty(); ++n) {
        for (Problem& pb : problems) pb.n = n;
        std::vector<Fit> best;
        if ((rc = run_fits(p, problems, d_sim, best))) return rc;
        std::vector<int> next_active;
        std::vector<Problem> next_problems;
        for (size_t i = 0; i < active.size(); ++i) {
            if (any_overlap(best[i], n, z)) continue;                  // n - 1 components stay (the fit already held)
            chosen[active[i]] = best[i];
            n_components[active[i]] = n;
            next_active.push_back(active[i]);
            next_problems.push_back(problems[i]);
        }
        active.swap(next_active);
        problems.swap(next_problems);
    }

    // ---- labels of the trimmed sizes under the chosen mixture (predict / predict_proba, split_alleles.py:258-279)
    for (int g = 0; g < n_regions; ++g) {
        const int n = n_components[g];
        if (n == 0) continue;
        const Fit& f = chosen[g];
        double c0[kMaxC], pc[kMaxC];
        for (int j = 0; j < n; ++j) {
            weights[(size_t)g * C + j] = f.w[j]; means[(size_t)g * C + j] = f.m[j]; variances[(size_t)g * C + j] = f.v[j];
            pc[j] = 1.0 / sqrt(f.v[j]);
            c0[j] = log(pc[j]) + log(f.w[j]) - 0.5 * kLog2Pi;
        }
        for (long long t = toff[g]; t < toff[g + 1]; ++t) {
            double lp[kMaxC], top = -INFINITY;
            int lab = 0;
            for (int j = 0; j < n; ++j) {
                const double d = (kept[t] - f.m[j]) * pc[j];
                lp[j] = c0[j] - 0.5 * d * d;
                if (lp[j] > top) { top = lp[j]; lab = j; }
            }
            double s = 0;
            for (int j = 0; j < n; ++j) s += exp(lp[j] - top);
            label[kept_src[t]] = lab;
            proba[kept_src[t]] = 1.0 / s;              // exp(lp[lab] - (top + log s))
        }
    }
    return NR_OK;
}
