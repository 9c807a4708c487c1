"""CPU restatement of the mixture fits of one or two features (TEST INFRASTRUCTURE ONLY: tests/ and tools/).

What nr_gmm_fit (nanorepeat_b200/csrc/nr_gmm_nd.cu, kernel in nr_launch_gmm_nd.cu) computes for one problem:

    em_fit            <- sklearn.mixture.GaussianMixture(covariance_type='diag').fit from explicit starting parameters:
                         the E / M steps and the stopping rule of BaseMixture.fit_predict (scikit-learn 1.9), with D
                         features -- E step  sum_d [-1/2 (log 2 pi + ((x_d - mu_d) pc_d)^2) + log pc_d] + log w,
                         pc = 1 / sqrt(var); M step  nk = sum r + 10 eps, mu_d = sum r x_d / nk,
                         var_d = sum r x_d^2 / nk - mu_d^2 + reg_covar, w = nk / n_samples
    start_parameters  <- the library's stand-in for scikit-learn's k-means start; at D = 1 exactly
                         oracle/gmm.py:start_parameters
    best_fit          <- the best of n_init starts by lower bound (the first of the highest, scikit-learn's `>`),
                         components in the fit's order (not sorted)

Pinned: em_fit against scikit-learn itself from identical starts (tests/test_oracle_gmm_nd.py, 1e-9 relative), the
start rule at D = 1 against oracle/gmm.py.  The random draws (`key`) are oracle/gmm.py's, which the kernels share.
"""
import numpy as np

from .gmm import LOG_2PI, key, mix64  # noqa: F401  (mix64: the generator key is built on)

EPS10 = 10 * np.finfo(np.float64).eps


def _rows(x):
    x = np.asarray(x, dtype=np.float64)
    return x.reshape(-1, 1) if x.ndim == 1 else x


def m_step(x, resp, reg_covar=1e-6):
    """sklearn _estimate_gaussian_parameters, 'diag' -> (weights nk / n_samples, means (n, D), variances (n, D))"""
    x = _rows(x)
    nk = resp.sum(axis=0) + EPS10
    means = resp.T @ x / nk[:, None]
    var = resp.T @ (x * x) / nk[:, None] - means ** 2 + reg_covar
    return nk / len(x), means, var


def e_step(x, weights, means, var):
    """-> (mean log-likelihood, log responsibilities (N, n))"""
    x = _rows(x)
    pc = 1.0 / np.sqrt(np.asarray(var, dtype=np.float64))
    means = np.asarray(means, dtype=np.float64)
    d = (x[:, None, :] - means[None, :, :]) * pc[None, :, :]
    lp = (-0.5 * (LOG_2PI + d * d) + np.log(pc)[None, :, :]).sum(axis=2) + np.log(np.asarray(weights, dtype=np.float64))[None, :]
    top = lp.max(axis=1)
    norm = top + np.log(np.exp(lp - top[:, None]).sum(axis=1))
    return float(norm.mean()), lp - norm[:, None]


def em_fit(x, weights, means, var, tol=1e-3, max_iter=100, reg_covar=1e-6):
    """-> (weights, means (n, D), variances (n, D), lower bound, iterations, converged)"""
    x = _rows(x)
    weights = np.asarray(weights, dtype=np.float64)
    means, var = _rows(means).reshape(len(weights), -1), _rows(var).reshape(len(weights), -1)
    lower, converged, it = -np.inf, False, 0
    for it in range(1, max_iter + 1):
        prev = lower
        lower, log_resp = e_step(x, weights, means, var)
        weights, means, var = m_step(x, np.exp(log_resp), reg_covar)
        if abs(lower - prev) < tol:
            converged = True
            break
    return weights, means, var, lower, it, converged


def start_parameters(x, n, init, seed, region, lloyd=10, reg_covar=1e-6):
    """init 0 spreads the means evenly along the bounding box, lo_d + (j + 1/2) / n (hi_d - lo_d); the others take the
    sample rows key(seed, region, 1000 + 32 n + init, j) mod N; `lloyd` rounds of k-means on the squared Euclidean distance
    (|x - m| at D = 1, the same order; first index on a tie); then sklearn's own first M step on the one-hot labels."""
    x = _rows(x)
    N = len(x)
    if init == 0:
        lo, hi = x.min(axis=0), x.max(axis=0)
        means = np.array([lo + (j + 0.5) / n * (hi - lo) for j in range(n)])
    else:
        means = np.array([x[key(seed, region, 1000 + 32 * n + init, j) % N] for j in range(n)])

    def nearest(means):
        if x.shape[1] == 1:
            return np.argmin(np.abs(x[:, :1] - means[None, :, 0]), axis=1)
        return np.argmin(((x[:, None, :] - means[None, :, :]) ** 2).sum(axis=2), axis=1)

    for _ in range(lloyd):
        lab = nearest(means)
        for j in range(n):
            if np.any(lab == j):
                means[j] = x[lab == j].sum(axis=0) / np.count_nonzero(lab == j)
    lab = nearest(means)
    resp = np.zeros((N, n))
    resp[np.arange(N), lab] = 1.0
    return m_step(x, resp, reg_covar)


def best_fit(x, n, seed, region, n_init=10, tol=1e-3, max_iter=100, reg_covar=1e-6):
    """nr_gmm_fit with the k-means stand-in: best of n_init starts -> em_fit's tuple, components in the fit's order"""
    best = None
    for init in range(n_init):
        fit = em_fit(x, *start_parameters(x, n, init, seed, region, reg_covar=reg_covar), tol=tol, max_iter=max_iter,
                     reg_covar=reg_covar)
        if best is None or fit[3] > best[3]:
            best = fit
    return best


def predict(x, weights, means, var):
    return np.argmax(e_step(x, weights, means, var)[1], axis=1)
