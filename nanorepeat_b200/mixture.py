"""GaussianMixture: scikit-learn's class of that name for one or two features and covariance_type='diag', fitted on the GPU.

The reference's allele phasing fits sklearn.mixture.GaussianMixture(n, covariance_type='diag', n_init=10) to the
bootstrapped sizes of one repeat (split_alleles.py auto_GMM_1d) or of two (the joint CLI's 2-D phasing), for n = 1, 2, ...
until two components overlap.  This class keeps that interface and runs the fits through nr_gmm_fit
(include/nanorepeat_b200.h): the same EM in fp64, the same stopping rule, regularisation and choice among the starts.
What differs is where the starts come from: scikit-learn's k-means is replaced by the library's seeded k-means stand-in
(oracle/gmm_nd.py).  From explicit weights_init / means_init / precisions_init the fit is scikit-learn's to rounding.
predict, predict_proba, score_samples, score, bic and aic are scikit-learn's formulas on the fitted parameters.

    from nanorepeat_b200 import mixture
    mixture.install(split_alleles)      # the module's GaussianMixture (or its sklearn `mixture`) now fits on the GPU

Anything the GPU fit does not cover raises ValueError; there is no CPU fallback.
"""
import math
import types
import warnings

import numpy as np

from . import engine

MAX_FEATURES = 2


class NotFittedError(ValueError, AttributeError):
    """The estimator is used before fit (scikit-learn's exception of the same name derives from the same two)."""


try:                                  # the warning category scikit-learn users filter on, when scikit-learn is installed
    from sklearn.exceptions import ConvergenceWarning
except ImportError:                   # pragma: no cover
    class ConvergenceWarning(UserWarning):
        pass


def _as_samples(X, name="GaussianMixture", min_samples=1):
    """scikit-learn's check_array for this class: 2-D, numeric, finite, at least min_samples rows, at least one feature."""
    X = np.asarray(X)
    if X.ndim != 2:
        raise ValueError(f"Expected 2D array, got {'scalar' if X.ndim == 0 else str(X.ndim) + 'D'} array instead:\narray={X}.\n"
                         "Reshape your data either using array.reshape(-1, 1) if your data has a single feature or "
                         "array.reshape(1, -1) if it contains a single sample.")
    X = np.ascontiguousarray(X, dtype=np.float64)
    if np.isnan(X).any():
        raise ValueError(f"Input X contains NaN.\n{name} does not accept missing values encoded as NaN natively.")
    if not np.isfinite(X).all():
        raise ValueError("Input X contains infinity or a value too large for dtype('float64').")
    if X.shape[0] < min_samples:
        raise ValueError(f"Found array with {X.shape[0]} sample(s) (shape={X.shape}) while a minimum of {min_samples} is "
                         f"required by {name}.")
    if X.shape[1] < 1:
        raise ValueError(f"Found array with 0 feature(s) (shape={X.shape}) while a minimum of 1 is required by {name}.")
    return X


def _logsumexp(a):
    top = a.max(axis=1)
    with np.errstate(divide="ignore"):
        return np.log(np.exp(a - top[:, None]).sum(axis=1)) + top


class GaussianMixture:
    """sklearn.mixture.GaussianMixture (same arguments, methods and fitted attributes) for covariance_type='diag' and one or
    two features, fitted by the library's CUDA kernel.  init_params='kmeans' uses the library's k-means stand-in, seeded
    from random_state (None: a seed drawn from numpy's global generator, so numpy.random.seed seeds the fits)."""

    def __init__(self, n_components=1, *, covariance_type="full", tol=1e-3, reg_covar=1e-6, max_iter=100, n_init=1,
                 init_params="kmeans", weights_init=None, means_init=None, precisions_init=None, random_state=None,
                 warm_start=False, verbose=0, verbose_interval=10):
        self.n_components = n_components
        self.covariance_type = covariance_type
        self.tol = tol
        self.reg_covar = reg_covar
        self.max_iter = max_iter
        self.n_init = n_init
        self.init_params = init_params
        self.weights_init = weights_init
        self.means_init = means_init
        self.precisions_init = precisions_init
        self.random_state = random_state
        self.warm_start = warm_start
        self.verbose = verbose
        self.verbose_interval = verbose_interval

    def get_params(self, deep=True):
        return {k: getattr(self, k) for k in ("n_components", "covariance_type", "tol", "reg_covar", "max_iter", "n_init",
                                              "init_params", "weights_init", "means_init", "precisions_init", "random_state",
                                              "warm_start", "verbose", "verbose_interval")}

    def set_params(self, **params):
        for k, v in params.items():
            if k not in self.get_params():
                raise ValueError(f"Invalid parameter {k!r} for estimator {self!r}.")
            setattr(self, k, v)
        return self

    def __repr__(self):
        return f"GaussianMixture(n_components={self.n_components}, covariance_type={self.covariance_type!r})"

    # ---- parameters
    def _check_parameters(self, X):
        def integral(name, lo):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or v < lo:
                raise ValueError(f"The '{name}' parameter of GaussianMixture must be an int in the range [{lo}, inf). Got {v!r} instead.")

        def real(name):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or not v >= 0:
                raise ValueError(f"The '{name}' parameter of GaussianMixture must be a float in the range [0.0, inf). Got {v!r} instead.")

        integral("n_components", 1)
        integral("n_init", 1)
        integral("max_iter", 0)
        integral("verbose_interval", 1)
        real("tol")
        real("reg_covar")
        if self.covariance_type not in ("full", "tied", "diag", "spherical"):
            raise ValueError("The 'covariance_type' parameter of GaussianMixture must be a str among {'diag', 'full', 'spherical', "
                             f"'tied'}}. Got {self.covariance_type!r} instead.")
        if self.init_params not in ("kmeans", "k-means++", "random", "random_from_data"):
            raise ValueError("The 'init_params' parameter of GaussianMixture must be a str among {'k-means++', 'kmeans', 'random', "
                             f"'random_from_data'}}. Got {self.init_params!r} instead.")
        # what the GPU fit covers (no CPU fallback)
        if self.covariance_type != "diag":
            raise ValueError(f"nanorepeat_b200.mixture.GaussianMixture fits covariance_type='diag' only, not {self.covariance_type!r}")
        if self.init_params != "kmeans":
            raise ValueError(f"nanorepeat_b200.mixture.GaussianMixture starts from init_params='kmeans' (its k-means stand-in) or "
                             f"explicit parameters only, not {self.init_params!r}")
        if self.warm_start:
            raise ValueError("nanorepeat_b200.mixture.GaussianMixture does not support warm_start=True")
        if self.max_iter < 1:
            raise ValueError("nanorepeat_b200.mixture.GaussianMixture needs max_iter >= 1")
        if self.n_components > engine.GMM_MAX_COMPONENTS:
            raise ValueError(f"nanorepeat_b200.mixture.GaussianMixture fits at most {engine.GMM_MAX_COMPONENTS} components, "
                             f"not {self.n_components}")
        if self.n_init > 64:
            raise ValueError("nanorepeat_b200.mixture.GaussianMixture runs at most 64 starts (n_init <= 64)")
        n, D = self.n_components, X.shape[1]
        if D > MAX_FEATURES:
            raise ValueError(f"nanorepeat_b200.mixture.GaussianMixture fits one or two features, not {D}")
        given = [v is not None for v in (self.weights_init, self.means_init, self.precisions_init)]
        inits = None
        if any(given):
            if not all(given):
                raise ValueError("nanorepeat_b200.mixture.GaussianMixture needs weights_init, means_init and precisions_init "
                                 "together (scikit-learn completes a partial start from its own k-means)")
            w = np.asarray(self.weights_init, dtype=np.float64)
            m = np.asarray(self.means_init, dtype=np.float64)
            p = np.asarray(self.precisions_init, dtype=np.float64)
            if w.shape != (n,):
                raise ValueError(f"The parameter 'weights' should have the shape of {(n,)}, but got {w.shape}")
            if np.any(w < 0.0) or np.any(w > 1.0):
                raise ValueError("The parameter 'weights' should be in the range [0, 1], but got max value %.5f, min value %.5f"
                                 % (w.max(), w.min()))
            if not np.allclose(abs(1.0 - w.sum()), 0.0, atol=1e-8):
                raise ValueError("The parameter 'weights' should be normalized, but got sum(weights) = %.5f" % w.sum())
            if m.shape != (n, D):
                raise ValueError(f"The parameter 'means' should have the shape of {(n, D)}, but got {m.shape}")
            if p.shape != (n, D):
                raise ValueError(f"The parameter 'diag precisions' should have the shape of {(n, D)}, but got {p.shape}")
            if np.any(p <= 0.0):
                raise ValueError("'diag precision' should be positive")
            inits = (w, m, p)
        return inits

    def _seed(self):
        rs = self.random_state
        if rs is None or rs is np.random:
            return int(np.random.randint(0, np.iinfo(np.int64).max, dtype=np.int64))
        if isinstance(rs, (int, np.integer)) and not isinstance(rs, bool):
            return int(rs) & ((1 << 64) - 1)
        if isinstance(rs, np.random.RandomState):
            return int(rs.randint(0, np.iinfo(np.int64).max, dtype=np.int64))
        raise ValueError(f"{rs!r} cannot be used to seed a numpy.random.RandomState instance")

    # ---- fit
    def fit(self, X, y=None):
        self.fit_predict(X, y)
        return self

    def fit_predict(self, X, y=None):
        X = _as_samples(X, min_samples=2)
        if X.shape[0] < self.n_components:
            raise ValueError("Expected n_samples >= n_components "
                             f"but got n_components = {self.n_components}, n_samples = {X.shape[0]}")
        inits = self._check_parameters(X)
        n, D = int(self.n_components), X.shape[1]
        params = engine.GmmParams(max_components=n, n_init=int(self.n_init), max_iter=int(self.max_iter), tol=float(self.tol),
                                  reg_covar=float(self.reg_covar), seed=self._seed())
        init = None if inits is None else ([inits[0]], [inits[1]], [inits[2]])
        r = engine.gmm_fit(params, [X], [n], D, init=init)
        w, m, v = r["weights"][0].copy(), r["means"][0].reshape(n, D).copy(), r["variances"][0].reshape(n, D).copy()
        if not (np.all(np.isfinite(v)) and np.all(v > 0)):
            raise ValueError("Fitting the mixture model failed because some components have ill-defined empirical covariance "
                             "(for instance caused by singleton or collapsed samples). Try to decrease the number of "
                             "components, increase reg_covar, or scale the input data.")
        self.weights_ = w / w.sum()                   # scikit-learn's M step normalises by the sum of nk
        self.means_ = m
        self.covariances_ = v
        self.precisions_cholesky_ = 1.0 / np.sqrt(v)
        self.precisions_ = self.precisions_cholesky_ ** 2
        self.converged_ = bool(r["converged"][0])
        self.n_iter_ = int(r["iters"][0])
        self.lower_bound_ = float(r["lower"][0])
        self.n_features_in_ = D
        if self.verbose:
            print(f"Initialization {'converged' if self.converged_ else 'did not converge'}. lower bound {self.lower_bound_:.5f}.")
        if not self.converged_:
            warnings.warn("Best performing initialization did not converge. Try different init parameters, or increase "
                          "max_iter, tol, or check for degenerate data.", ConvergenceWarning)
        return self.predict(X)

    # ---- scoring (scikit-learn's formulas, _estimate_log_gaussian_prob for 'diag')
    def _check_fitted(self, X):
        if not hasattr(self, "means_"):
            raise NotFittedError("This GaussianMixture instance is not fitted yet. Call 'fit' with appropriate arguments "
                                 "before using this estimator.")
        X = _as_samples(X)
        if X.shape[1] != self.n_features_in_:
            raise ValueError(f"X has {X.shape[1]} features, but GaussianMixture is expecting {self.n_features_in_} features as input.")
        return X

    def _estimate_weighted_log_prob(self, X):
        pc = self.precisions_cholesky_
        precisions = pc ** 2
        log_prob = (np.sum(self.means_ ** 2 * precisions, axis=1) - 2.0 * (X @ (self.means_ * precisions).T)
                    + (X ** 2) @ precisions.T)
        log_det = np.sum(np.log(pc), axis=1)
        return -0.5 * (X.shape[1] * math.log(2 * math.pi) + log_prob) + log_det + np.log(self.weights_)

    def score_samples(self, X):
        return _logsumexp(self._estimate_weighted_log_prob(self._check_fitted(X)))

    def score(self, X, y=None):
        return float(np.mean(self.score_samples(X)))

    def predict(self, X):
        return np.argmax(self._estimate_weighted_log_prob(self._check_fitted(X)), axis=1)

    def predict_proba(self, X):
        wlp = self._estimate_weighted_log_prob(self._check_fitted(X))
        with np.errstate(under="ignore"):
            return np.exp(wlp - _logsumexp(wlp)[:, None])

    def _n_parameters(self):
        n, D = self.means_.shape
        return int(n * D + n * D + n - 1)

    def bic(self, X):
        X = np.asarray(X)
        return -2 * self.score(X) * X.shape[0] + self._n_parameters() * math.log(X.shape[0])

    def aic(self, X):
        X = np.asarray(X)
        return -2 * self.score(X) * X.shape[0] + 2 * self._n_parameters()


class _MixtureNamespace(types.SimpleNamespace):
    """Stands in for a module's `mixture` (scikit-learn's submodule): GaussianMixture is this module's class, every other
    name is looked up in the module it replaced."""

    def __init__(self, replaced):
        super().__init__(GaussianMixture=GaussianMixture)
        object.__setattr__(self, "_replaced", replaced)

    def __getattr__(self, name):
        return getattr(object.__getattribute__(self, "_replaced"), name)


def install(module):
    """Make `module` fit its mixtures on the GPU.  A module that holds GaussianMixture (`from sklearn.mixture import
    GaussianMixture`) gets this class in its place; one that holds scikit-learn's `mixture` submodule (`from sklearn import
    mixture`) gets a namespace whose GaussianMixture is this class.  scikit-learn itself is not touched.  Returns what was
    replaced (put it back with setattr to undo)."""
    if hasattr(module, "GaussianMixture"):
        old = module.GaussianMixture
        module.GaussianMixture = GaussianMixture
        return old
    if hasattr(module, "mixture"):
        old = module.mixture
        module.mixture = _MixtureNamespace(old)
        return old
    raise ValueError(f"{getattr(module, '__name__', module)!r} holds neither GaussianMixture nor a `mixture` module")
