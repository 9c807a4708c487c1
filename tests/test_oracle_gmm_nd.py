"""oracle/gmm_nd.py (the CPU restatement of nr_gmm_fit) against scikit-learn itself: EM from identical explicit starts at one
and two features, and the start rule against oracle/gmm.py at one feature."""
import random
import warnings

import numpy as np
import pytest

from oracle import gmm, gmm_nd


def _blobs(rng, n, D, per=(60, 300)):
    """n clusters of D features, apart from each other."""
    x = []
    for j in range(n):
        c = [rng.uniform(5, 200) for _ in range(D)]
        s = [rng.uniform(0.5, 4.0) for _ in range(D)]
        x += [[c[d] + rng.gauss(0, s[d]) for d in range(D)] for _ in range(rng.randint(*per))]
    rng.shuffle(x)
    return np.array(x)


def _start(rng, x, n):
    D = x.shape[1]
    w0 = np.array([rng.uniform(0.5, 1.5) for _ in range(n)])
    w0 /= w0.sum()
    m0 = x[rng.sample(range(len(x)), n)] + np.array([[rng.uniform(-1, 1) for _ in range(D)] for _ in range(n)])
    p0 = 1.0 / (x.var(axis=0)[None, :] / n * np.array([[rng.uniform(0.5, 2.0) for _ in range(D)] for _ in range(n)]))
    return w0, m0, p0


@pytest.mark.parametrize("D", [1, 2])
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6])
def test_em_equals_sklearn_from_the_same_start(D, n):
    from sklearn.mixture import GaussianMixture
    rng = random.Random(100 * D + n)
    for case in range(3):
        x = _blobs(rng, max(n, rng.choice([n, n + 1])), D)
        w0, m0, p0 = _start(rng, x, n)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            sk = GaussianMixture(n_components=n, covariance_type="diag", n_init=1, weights_init=w0, means_init=m0,
                                 precisions_init=p0).fit(x)
        w, m, v, lower, it, conv = gmm_nd.em_fit(x, w0, m0, 1.0 / p0)
        assert it == sk.n_iter_ and conv == sk.converged_, (case, it, sk.n_iter_)
        assert np.allclose(w, sk.weights_, rtol=1e-9, atol=0), case
        assert np.allclose(m, sk.means_, rtol=1e-9, atol=0), case
        assert np.allclose(v, sk.covariances_, rtol=1e-9, atol=0), case
        assert abs(lower - sk.lower_bound_) <= 1e-9 * abs(sk.lower_bound_), (case, lower, sk.lower_bound_)
        assert np.array_equal(gmm_nd.predict(x, w, m, v), sk.predict(x)), case


def test_one_feature_em_equals_the_1d_checker():
    rng = random.Random(3)
    x = _blobs(rng, 3, 1)
    w0, m0, p0 = _start(rng, x, 3)
    a = gmm_nd.em_fit(x, w0, m0, 1.0 / p0)
    b = gmm.em_fit(x[:, 0], w0, m0[:, 0], 1.0 / p0[:, 0])
    assert a[4:] == b[4:]
    for u, t in zip(a[:4], b[:4]):
        assert np.allclose(np.ravel(u), np.ravel(t), rtol=1e-9, atol=0)     # E steps: (x - m) pc here, x pc - m pc there


@pytest.mark.parametrize("n", [1, 2, 3, 5])
def test_start_rule_at_one_feature_is_the_1d_start(n):
    rng = random.Random(n)
    x = _blobs(rng, 3, 1)[:, 0]
    for init in range(6):
        a = gmm_nd.start_parameters(x, n, init, seed=9, region=4)
        b = gmm.start_parameters(x, n, init, seed=9, region=4)
        assert np.allclose(a[0], b[0], rtol=1e-13, atol=0), init
        assert np.allclose(a[1][:, 0], b[1], rtol=1e-13, atol=0), init
        assert np.allclose(a[2][:, 0], b[2], rtol=1e-12, atol=0), init


def test_start_rule_at_two_features():
    """start 0: means evenly along the bounding box's diagonal before the Lloyd rounds; the others: hashed sample rows"""
    rng = random.Random(5)
    x = _blobs(rng, 3, 2)
    w, m, v = gmm_nd.start_parameters(x, 3, 0, seed=1, region=2, lloyd=0)
    lo, hi = x.min(axis=0), x.max(axis=0)
    lab = np.argmin(((x[:, None, :] - (lo + (np.arange(3)[:, None] + 0.5) / 3 * (hi - lo))[None]) ** 2).sum(axis=2), axis=1)
    assert np.allclose(w, np.bincount(lab, minlength=3) / len(x))
    rows = [gmm.key(1, 2, 1000 + 32 * 3 + 4, j) % len(x) for j in range(3)]
    resp = np.zeros((len(x), 3))
    resp[np.arange(len(x)), np.argmin(((x[:, None, :] - x[rows][None]) ** 2).sum(axis=2), axis=1)] = 1
    assert np.allclose(gmm_nd.start_parameters(x, 3, 4, seed=1, region=2, lloyd=0)[1], gmm_nd.m_step(x, resp)[1], rtol=1e-12)
    # best_fit keeps the fit's component order and picks the first of the highest lower bounds
    fit = gmm_nd.best_fit(x, 3, seed=1, region=2, n_init=4)
    fits = [gmm_nd.em_fit(x, *gmm_nd.start_parameters(x, 3, s, 1, 2)) for s in range(4)]
    b = max(range(4), key=lambda s: (fits[s][3], -s))
    assert np.array_equal(fit[1], fits[b][1]) and fit[3] == fits[b][3]
