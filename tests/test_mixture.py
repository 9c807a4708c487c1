"""nanorepeat_b200.mixture.GaussianMixture without a GPU: its scoring against scikit-learn's on the same parameters, its
argument checks against scikit-learn's errors, and install() on modules of both shapes."""
import types
import warnings

import numpy as np
import pytest

from nanorepeat_b200 import mixture


def _fitted_pair(D, n, seed):
    """a scikit-learn GaussianMixture fitted on blobs, and this class holding the same parameters"""
    from sklearn.mixture import GaussianMixture
    rng = np.random.default_rng(seed)
    x = np.concatenate([rng.normal(rng.uniform(0, 100, D), rng.uniform(0.5, 3, D), size=(rng.integers(50, 200), D)) for _ in range(n)])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sk = GaussianMixture(n_components=n, covariance_type="diag", random_state=seed).fit(x)
    ours = mixture.GaussianMixture(n_components=n, covariance_type="diag")
    ours.weights_, ours.means_, ours.covariances_ = sk.weights_.copy(), sk.means_.copy(), sk.covariances_.copy()
    ours.precisions_cholesky_ = 1.0 / np.sqrt(ours.covariances_)
    ours.precisions_ = ours.precisions_cholesky_ ** 2
    ours.n_features_in_ = D
    return sk, ours, x


@pytest.mark.parametrize("D,n", [(1, 1), (1, 3), (2, 2), (2, 4)])
def test_scoring_equals_sklearn(D, n):
    sk, ours, x = _fitted_pair(D, n, 10 * D + n)
    y = x + np.random.default_rng(1).normal(0, 2, size=x.shape)
    for X in (x, y):
        assert np.array_equal(ours.predict(X), sk.predict(X))
        assert np.allclose(ours.predict_proba(X), sk.predict_proba(X), rtol=1e-12, atol=1e-300)
        assert np.allclose(ours.score_samples(X), sk.score_samples(X), rtol=1e-12, atol=0)
        assert abs(ours.score(X) - sk.score(X)) <= 1e-12 * abs(sk.score(X))
        assert abs(ours.bic(X) - sk.bic(X)) <= 1e-12 * abs(sk.bic(X))
        assert abs(ours.aic(X) - sk.aic(X)) <= 1e-12 * abs(sk.aic(X))
    assert np.allclose(ours.precisions_, sk.precisions_, rtol=1e-12) and np.allclose(ours.precisions_cholesky_, sk.precisions_cholesky_, rtol=1e-12)
    assert ours._n_parameters() == sk._n_parameters()


def _sk_error(make, X):
    from sklearn.mixture import GaussianMixture
    with pytest.raises(ValueError) as e:
        make(GaussianMixture).fit(X)
    return str(e.value)


@pytest.mark.parametrize("case", ["few_samples", "nan", "inf", "one_sample", "one_d", "weights_sum", "means_shape",
                                  "precision_sign", "n_components_zero", "tol_negative"])
def test_argument_errors_match_sklearn(case):
    x = np.arange(12, dtype=np.float64).reshape(6, 2)
    kw, X = dict(covariance_type="diag"), x
    if case == "few_samples":
        kw["n_components"] = 7
    elif case == "nan":
        X = x.copy(); X[3, 1] = np.nan
    elif case == "inf":
        X = x.copy(); X[0, 0] = np.inf
    elif case == "one_sample":
        X = x[:1]
    elif case == "one_d":
        X = x[:, 0]
    elif case == "weights_sum":
        kw.update(n_components=2, weights_init=[0.5, 0.6], means_init=[[0, 1], [5, 6]], precisions_init=[[1, 1], [1, 1]])
    elif case == "means_shape":
        kw.update(n_components=2, weights_init=[0.5, 0.5], means_init=[[0], [5]], precisions_init=[[1, 1], [1, 1]])
    elif case == "precision_sign":
        kw.update(n_components=2, weights_init=[0.5, 0.5], means_init=[[0, 1], [5, 6]], precisions_init=[[1, -1], [1, 1]])
    elif case == "n_components_zero":
        kw["n_components"] = 0
    elif case == "tol_negative":
        kw["tol"] = -1.0
    want = _sk_error(lambda cls: cls(**kw), X)
    with pytest.raises(ValueError) as e:
        mixture.GaussianMixture(**kw).fit(X)
    got = str(e.value)
    # the first line of scikit-learn's message (its later lines quote the array, whose printing differs)
    assert got.split("\n")[0] == want.split("\n")[0], (got, want)


@pytest.mark.parametrize("kw,X", [(dict(covariance_type="full"), np.zeros((5, 2))), (dict(covariance_type="diag"), np.zeros((5, 3))),
                                  (dict(covariance_type="diag", warm_start=True), np.zeros((5, 2))),
                                  (dict(covariance_type="diag", init_params="random"), np.zeros((5, 2))),
                                  (dict(covariance_type="diag", n_components=33), np.zeros((40, 2))),
                                  (dict(covariance_type="diag", n_components=2, means_init=[[0, 0], [1, 1]]), np.zeros((5, 2)))])
def test_what_the_gpu_fit_does_not_cover_raises(kw, X):
    with pytest.raises(ValueError, match="nanorepeat_b200"):
        mixture.GaussianMixture(**kw).fit(X + np.arange(len(X))[:, None])


def test_not_fitted_and_feature_count():
    g = mixture.GaussianMixture(covariance_type="diag")
    with pytest.raises(mixture.NotFittedError):
        g.predict(np.zeros((3, 1)))
    _sk, ours, _x = _fitted_pair(2, 2, 3)
    with pytest.raises(ValueError, match="X has 1 features, but GaussianMixture is expecting 2 features"):
        ours.predict(np.zeros((3, 1)))


def test_random_state_none_draws_from_numpy():
    g = mixture.GaussianMixture(covariance_type="diag")
    np.random.seed(5)
    a = g._seed()
    np.random.seed(5)
    assert g._seed() == a
    assert mixture.GaussianMixture(random_state=17)._seed() == 17
    assert mixture.GaussianMixture(random_state=np.random.RandomState(2))._seed() == mixture.GaussianMixture(random_state=np.random.RandomState(2))._seed()


def test_install_on_both_module_shapes():
    import sklearn.mixture
    from sklearn.mixture import GaussianMixture as SkGM
    a = types.ModuleType("split_alleles_a")          # `from sklearn.mixture import GaussianMixture`
    a.GaussianMixture = SkGM
    assert mixture.install(a) is SkGM and a.GaussianMixture is mixture.GaussianMixture
    b = types.ModuleType("split_alleles_b")          # `from sklearn import mixture`
    b.mixture = sklearn.mixture
    assert mixture.install(b) is sklearn.mixture
    assert b.mixture.GaussianMixture is mixture.GaussianMixture
    assert b.mixture.BayesianGaussianMixture is sklearn.mixture.BayesianGaussianMixture
    assert sklearn.mixture.GaussianMixture is SkGM                           # scikit-learn itself is untouched
    with pytest.raises(ValueError):
        mixture.install(types.ModuleType("neither"))


def test_get_and_set_params_follow_sklearn():
    from sklearn.mixture import GaussianMixture
    assert set(mixture.GaussianMixture().get_params()) == set(GaussianMixture().get_params())
    g = mixture.GaussianMixture().set_params(n_components=3, covariance_type="diag")
    assert g.n_components == 3 and g.covariance_type == "diag"
