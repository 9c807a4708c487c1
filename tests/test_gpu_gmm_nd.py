"""GPU parity of the mixture fits of one or two features (nr_gmm_fit; csrc/nr_launch_gmm_nd.cu) with the CPU checker that
shares its random draws (oracle/gmm_nd.py, itself pinned to scikit-learn in tests/test_oracle_gmm_nd.py), with the 1-D fit
(nr_gmm1d_fit), and of nanorepeat_b200.mixture.GaussianMixture with scikit-learn itself.  Tolerances are written at each
check: the device and the checker sum in different orders, nothing else differs."""
import math
import random
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _blobs(rng, centers, sds, counts):
    x = []
    for c, s, k in zip(centers, sds, counts):
        x += [[ci + rng.gauss(0, si) for ci, si in zip(c, s)] for _ in range(k)]
    rng.shuffle(x)
    return np.array(x)


def _problems(seed, D, n_problems, per=(150, 600), max_n=6):
    rng = random.Random(seed)
    data, ncs = [], []
    for _ in range(n_problems):
        k = rng.randint(1, 4)
        centers = [[rng.uniform(5, 150) for _ in range(D)] for _ in range(k)]
        sds = [[rng.uniform(0.5, 4) for _ in range(D)] for _ in range(k)]
        data.append(_blobs(rng, centers, sds, [rng.randint(*per) for _ in range(k)]))
        ncs.append(min(max_n, rng.choice([k, k, max(1, k - 1), k + 1])))
    return data, ncs


def _close(a, b, rtol):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b)) + 1e-300))


def _equal_checker(got, i, exp, x, rtol=1e-7):
    w, m, v, lower, it, conv = exp
    assert got["iters"][i] == it and bool(got["converged"][i]) == conv, (i, got["iters"][i], it)
    assert abs(got["lower"][i] - lower) <= rtol * abs(lower), (i, got["lower"][i], lower)
    D = x.shape[1]
    gw, gm, gv = got["weights"][i], got["means"][i].reshape(-1, D), got["variances"][i].reshape(-1, D)
    assert _close(gw, w, rtol) and _close(gm, m, rtol) and _close(gv, v, 10 * rtol), (i, gw, w, gm, m)
    from oracle import gmm_nd
    assert np.array_equal(gmm_nd.predict(x, gw, gm, gv), gmm_nd.predict(x, w, m, v)), i


@pytest.mark.parametrize("D", [1, 2])
def test_kmeans_starts_equal_checker_on_the_block_path(engine, D):
    from oracle import gmm_nd
    data, ncs = _problems(10 + D, D, 8)
    p = engine.GmmParams(seed=31, max_components=8, n_init=10)
    got = engine.gmm_fit(p, data, ncs, D, region_ids=list(range(40, 48)))
    st = engine.last_stats()
    assert st["n_tasks"] == 80 and st["kernel_launches"] == 1
    for i, x in enumerate(data):
        _equal_checker(got, i, gmm_nd.best_fit(x, ncs[i], 31, 40 + i, n_init=10), x)


@pytest.mark.parametrize("D", [1, 2])
def test_explicit_starts_equal_checker_and_keep_their_order(engine, D):
    from oracle import gmm_nd
    rng = random.Random(D)
    data, ncs = _problems(20 + D, D, 6)
    inits = ([], [], [])
    for x, n in zip(data, ncs):
        w0 = np.full(n, 1.0 / n)
        m0 = x[rng.sample(range(len(x)), n)][::-1].copy()
        p0 = np.tile(1.0 / (x.var(axis=0) / n), (n, 1))
        inits[0].append(w0); inits[1].append(m0); inits[2].append(p0)
    p = engine.GmmParams(seed=0, max_components=6, n_init=10)
    got = engine.gmm_fit(p, data, ncs, D, init=inits)
    assert engine.last_stats()["n_tasks"] == len(data)              # one start per problem
    for i, x in enumerate(data):
        _equal_checker(got, i, gmm_nd.em_fit(x, inits[0][i], inits[1][i], 1.0 / inits[2][i]), x)


@pytest.mark.parametrize("D", [1, 2])
def test_cluster_path_and_many_components_equal_checker(engine, D):
    """Problems of 16 384 samples and more take a cluster of 8 thread blocks per start; n up to 32."""
    from oracle import gmm_nd
    rng = random.Random(50 + D)
    big = [_blobs(rng, [[20] * D, [60] * D], [[2.0] * D, [3.0] * D], [9000, 8000]),
           _blobs(rng, [[15 + 10 * k] * D for k in range(6)], [[1.0] * D] * 6, [3000] * 6)]
    many = _blobs(rng, [[rng.uniform(0, 300) for _ in range(D)] for _ in range(32)], [[1.0] * D] * 32, [40] * 32)
    data, ncs = big + [many, many[:2000]], [2, 6, 32, 20]
    p = engine.GmmParams(seed=5, max_components=32, n_init=3)
    got = engine.gmm_fit(p, data, ncs, D, region_ids=[7, 8, 9, 10])
    assert engine.last_stats()["kernel_launches"] == 2
    for i, x in enumerate(data):
        _equal_checker(got, i, gmm_nd.best_fit(x, ncs[i], 5, 7 + i, n_init=3), x)
    # explicit starts on the cluster path
    w0, m0 = np.array([0.5, 0.5]), big[0][:2].copy()
    p0 = np.tile(1.0 / big[0].var(axis=0), (2, 1))
    got = engine.gmm_fit(p, big[:1], [2], D, init=([w0], [m0], [p0]))
    _equal_checker(got, 0, gmm_nd.em_fit(big[0], w0, m0, 1.0 / p0), big[0])


def test_result_does_not_depend_on_the_other_problems(engine):
    data, ncs = _problems(70, 2, 6)
    data.append(_blobs(random.Random(1), [[30, 8], [55, 12]], [[2, 1], [3, 1]], [9000, 9000]))
    ncs.append(2)
    p = engine.GmmParams(seed=11, max_components=6)
    rid = list(range(100, 107))
    together = engine.gmm_fit(p, data, ncs, 2, region_ids=rid)
    for i in (0, 3, 6):
        alone = engine.gmm_fit(p, [data[i]], [ncs[i]], 2, region_ids=[rid[i]])
        assert alone["lower"][0] == together["lower"][i] and alone["iters"][0] == together["iters"][i]
        for k in ("weights", "means", "variances"):
            assert np.array_equal(alone[k][0], together[k][i]), (i, k)


def test_one_feature_equals_the_1d_fit(engine):
    """At D = 1 the kernel is fit_kernel's arithmetic with one loop level more (the feature); the 1-D fit sorts by mean."""
    data, ncs = _problems(80, 1, 10)
    data.append(_blobs(random.Random(2), [[20], [45]], [[2], [3]], [10000, 8000]))
    ncs.append(2)
    p = engine.GmmParams(seed=4, max_components=6)
    nd = engine.gmm_fit(p, data, ncs, 1, region_ids=list(range(10, 21)))
    one = engine.gmm1d_fit(p, [x[:, 0] for x in data], ncs, region_ids=list(range(10, 21)))
    for i in range(len(data)):
        assert nd["iters"][i] == one["iters"][i], i
        assert abs(nd["lower"][i] - one["lower"][i]) <= 1e-9 * abs(one["lower"][i]), i
        o = np.argsort(nd["means"][i][:, 0], kind="stable")
        assert _close(nd["weights"][i][o], one["weights"][i], 1e-9) and _close(nd["means"][i][o, 0], one["means"][i], 1e-9), i
        assert _close(nd["variances"][i][o, 0], one["variances"][i], 1e-9), i


def test_errors(engine):
    p = engine.GmmParams(max_components=4)
    x = np.arange(20, dtype=np.float64).reshape(10, 2)
    cases = [(lambda: engine.gmm_fit(p, [x], [2], 3), "n_features"),
             (lambda: engine.gmm_fit(p, [x[:1]], [2], 2), "fewer than"),
             (lambda: engine.gmm_fit(engine.GmmParams(max_components=33), [x], [2], 2), "max_components"),
             (lambda: engine.gmm_fit(p, [np.where(x == 7, np.nan, x)], [2], 2), "not finite")]
    for call, what in cases:
        with pytest.raises(engine.NanoRepeatB200Error, match=what) as e:
            call()
        assert e.value.code == -2


def test_class_equals_sklearn_from_explicit_starts(engine):
    from sklearn.mixture import GaussianMixture as SkGM
    from nanorepeat_b200.mixture import GaussianMixture
    rng = random.Random(6)
    for D in (1, 2):
        for n in (1, 2, 3, 5):
            x = _blobs(rng, [[rng.uniform(5, 150) for _ in range(D)] for _ in range(n)], [[rng.uniform(0.5, 3) for _ in range(D)]] * n,
                       [rng.randint(100, 400) for _ in range(n)])
            kw = dict(n_components=n, covariance_type="diag", weights_init=np.full(n, 1.0 / n),
                      means_init=x[rng.sample(range(len(x)), n)], precisions_init=np.tile(1.0 / x.var(axis=0), (n, 1)))
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                sk = SkGM(**kw).fit(x)
                ours = GaussianMixture(**kw)
                lab = ours.fit_predict(x)
            assert ours.n_iter_ == sk.n_iter_ and ours.converged_ == sk.converged_, (D, n)
            assert np.array_equal(lab, sk.predict(x)), (D, n)
            for a in ("weights_", "means_", "covariances_", "precisions_", "precisions_cholesky_"):
                assert _close(getattr(ours, a), getattr(sk, a), 1e-7), (D, n, a)
            assert abs(ours.lower_bound_ - sk.lower_bound_) <= 1e-7 * abs(sk.lower_bound_)
            assert ours.n_features_in_ == D


# ---- two-allele loci of two repeats (HTT-like: CAG and CCG sizes), phased the way the joint CLI's 2-D phasing does

def _locus(seed, reads_per_allele=(40, 35), error_rate=0.07):
    """reads' (CAG, CCG) sizes of two alleles, and their 100-fold bootstrap with noise sd = error_rate * (10 + size) per
    feature (DESIGN section 4.7)"""
    rng = np.random.default_rng(seed)
    sizes = np.concatenate([np.column_stack([rng.normal(17, 0.6, reads_per_allele[0]), rng.normal(10, 0.4, reads_per_allele[0])]),
                            np.column_stack([rng.normal(55, 1.5, reads_per_allele[1]), rng.normal(7, 0.4, reads_per_allele[1])])])
    truth = np.repeat([0, 1], reads_per_allele)
    sim = np.tile(sizes, (100, 1))
    sim = sim + error_rate * (10 + sim) * rng.standard_normal(sim.shape)
    return sizes, truth, sim


def _overlap_both(gm, z):
    """two components whose [mean -+ z sd] intervals (sd floored at 1) overlap in both features"""
    n = len(gm.weights_)
    for i in range(n):
        for j in range(i + 1, n):
            both = True
            for d in range(gm.means_.shape[1]):
                si, sj = max(1.0, math.sqrt(gm.covariances_[i, d])), max(1.0, math.sqrt(gm.covariances_[j, d]))
                lo = max(gm.means_[i, d] - z * si, gm.means_[j, d] - z * sj)
                hi = min(gm.means_[i, d] + z * si, gm.means_[j, d] + z * sj)
                both = both and lo - hi <= 0
            if both:
                return True
    return False


def _auto_n(cls, sim, z, seed, max_n=5):
    prev = None
    for n in range(1, max_n + 1):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            gm = cls(n_components=n, covariance_type="diag", n_init=10, random_state=seed).fit(sim)
        if n > 1 and _overlap_both(gm, z):
            return n - 1, prev
        prev = gm
    return max_n, prev


def test_two_repeat_loci_agree_with_sklearn(engine):
    from scipy.stats import norm
    from sklearn.mixture import GaussianMixture as SkGM
    from nanorepeat_b200.mixture import GaussianMixture
    z = norm.isf(0.15)
    for locus in range(6):
        sizes, truth, sim = _locus(1000 + locus)
        n_ours, ours = _auto_n(GaussianMixture, sim, z, locus)
        n_sk, sk = _auto_n(SkGM, sim, z, locus)
        assert n_ours == n_sk == 2, (locus, n_ours, n_sk)
        o, s = np.argsort(ours.means_[:, 0]), np.argsort(sk.means_[:, 0])
        rank_o, rank_s = np.argsort(o), np.argsort(s)
        lo, ls = rank_o[ours.predict(sizes)], rank_s[sk.predict(sizes)]
        assert np.count_nonzero(lo != ls) <= 1, (locus, np.nonzero(lo != ls))
        assert np.count_nonzero(lo != truth) <= 1, locus
        for a, b in zip(o, s):
            se = np.sqrt(ours.covariances_[a] / (ours.weights_[a] * len(sim)))
            assert np.all(np.abs(ours.means_[a] - sk.means_[b]) <= 6 * se), (locus, ours.means_[a], sk.means_[b], se)
