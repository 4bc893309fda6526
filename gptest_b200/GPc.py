"""Binary GP classification behind the names the reference's ``GPc.py`` sketches.

/root/reference/GPc.py is an unfinished fragment (SyntaxError at GPc.py:10; ``ClassifierLikelihood``
is declared with ``def``): it fixes the likelihood (``log Phi(y f)``, GPc.py:5-6), the link selector
(``'Logit'`` else probit, GPc.py:17-21), the label convention ({0,1} -> {-1,+1}, anything else is an
AssertionError, GPc.py:24-38) and cites Rasmussen & Williams eq. 3.12 (GPc.py:42-44).  This module
keeps those names and finishes the path the way the sibling ``GPpref.py`` is organised:
``ClassifierGaussianProcess(x_train, y_train, likelihood=..., delta_f=1e-6)`` with
``calc_laplace(loghyp, f=None) -> (f, lml)``, ``calc_nlml(loghyp)`` and ``predict``.
Newton mode finding (R&W Alg. 3.1), the evidence and the predictive distribution (Alg. 3.2) run on
the device through libgpb200; the specification the CUDA path is tested against is
``oracle/gpc_oracle.py`` (parity unpinned: there is no reference arithmetic).
"""
import numpy as np

from . import _lib


def _handle():
    return _lib.default_handle()


def std_norm_cdf(z):
    """scipy.special.ndtr as imported by GPc.py:2 (host helper for scalars / small arrays)."""
    from math import erfc, sqrt
    z = np.asarray(z, dtype=float)
    return np.vectorize(lambda v: 0.5 * erfc(-v / sqrt(2.0)))(z)


class NormCDF(object):
    """GPc.py:4-10."""

    def logpyf(self, y, f):
        return np.log(std_norm_cdf(y * f))                      # GPc.py:5-6

    def dlogpyf_df(self, y, f):
        """GPc.py:8-10 is cut off mid-expression; completed as y N(f)/Phi(y f) (R&W eq. 3.16)."""
        f = np.asarray(f, dtype=float)
        return y * np.exp(-0.5 * f * f) / np.sqrt(2 * np.pi) / std_norm_cdf(y * f)


def logistic_function(z):
    """GPc.py:13-14."""
    return 1.0 / (1 + np.exp(-z))


class ClassifierLikelihood(object):
    """GPc.py:16-55 (declared with ``def`` in the reference)."""

    def __init__(self, inverse_link_function=None):
        if inverse_link_function == 'Logit':                    # GPc.py:18-21
            self.inverse_link_function = logistic_function
            self.link_id = 1
        else:
            self.inverse_link_function = std_norm_cdf
            self.link_id = 0

    def _preprocess_values(self, Y):
        """GPc.py:24-38: labels must be {0,1} or {-1,1}; 0 becomes -1."""
        Y = np.asarray(Y)
        Y_prep = Y.astype(float).copy()
        Y1 = Y[Y.flatten() == 1].size
        Y2 = Y[Y.flatten() == 0].size
        Y3 = Y[Y.flatten() == -1].size
        assert ((Y1 + Y2 == Y.size) or (Y1 + Y3 == Y.size)), 'Inputs should be in {0,1} or {-1,1}.'
        Y_prep[Y.flatten() == 0] = -1
        return Y_prep

    def loglikelihood(self, y, f):
        """log p(y|f) under the chosen link (the first term of Psi, GPc.py:42-47)."""
        y = np.asarray(y, dtype=float)
        f = np.asarray(f, dtype=float)
        p = self.inverse_link_function(y * f)
        return np.log(np.clip(p, 1e-9, np.inf))                 # GPc.py:55


class ClassifierGaussianProcess(object):
    """The classifier GPc.py was heading for, shaped like PreferenceGaussianProcess (GPpref.py:96-161).

    loghyp = [log l_1 .. log l_D, log sigma_f]; f starts at 0; K gets the same jitter loop as
    GPpref.py:123-135; iteration stops when max|f_new - f| <= delta_f.
    """

    def __init__(self, x_train, y_train, likelihood=ClassifierLikelihood, delta_f=1e-6, max_iter=100,
                 inverse_link_function=None):
        x_train = np.asarray(x_train, dtype=float)
        self.x_train = x_train.reshape(len(x_train), -1)
        self._xdim = self.x_train.shape[1]
        self._nx = self.x_train.shape[0]
        self.likelihood = likelihood(inverse_link_function) if inverse_link_function else likelihood()
        self.y_train = self.likelihood._preprocess_values(np.asarray(y_train).reshape(-1))
        self.delta_f = delta_f
        self.max_iter = max_iter
        self.trace = None
        self.n_iter = 0
        self.jitter = None
        self._f_hat = None
        self._loghyp = None

    def _khyp(self, loghyp):
        loghyp = np.asarray(loghyp, dtype=float)
        return np.concatenate([np.exp(loghyp[0:self._xdim]), [np.exp(loghyp[self._xdim]) ** 2]])

    def calc_laplace(self, loghyp, f=None):
        """Mode f_hat (n,1) and the Laplace approximation of log p(y|X, theta)."""
        h = _handle()
        h.set_train(self.x_train)
        f0 = None if f is None else np.asarray(f, dtype=float).reshape(-1)
        fv, lml, iters, trace, jitter = h.gpc_laplace(self.y_train, self._khyp(loghyp), link=self.likelihood.link_id,
                                                      delta_f=self.delta_f, max_iter=self.max_iter, f0=f0)
        self.trace, self.n_iter, self.jitter = trace, iters, jitter
        self._f_hat, self._loghyp = fv, np.array(loghyp, dtype=float)
        return fv.reshape(-1, 1), lml

    def calc_nlml(self, loghyp):
        f, lml = self.calc_laplace(loghyp)
        return -lml

    def laplace_evidence_and_grad(self, loghyp, f0=None):
        """(lml, grad) for hyper-parameter fitting: the Laplace evidence ``calc_laplace`` returns and its exact
        gradient with respect to ``loghyp`` = [log l_1 .. log l_D, log sigma_f], with the fit's jitter held fixed
        (not in the reference).  The fit is ``calc_laplace(loghyp, f=f0)`` (same link, ``delta_f``, ``max_iter``); it
        must converge within ``max_iter``, otherwise the device refuses the gradient (``GpbError``).  ``f0``: start
        of the Newton iteration, e.g. the mode of the previous call (``self._f_hat``); ``predict`` at the same
        ``loghyp`` warm-starts from this fit.  Maximise the evidence, e.g.

            scipy.optimize.minimize(lambda t: tuple(-v for v in gp.laplace_evidence_and_grad(t, f0=gp._f_hat)),
                                    x0, jac=True, method='L-BFGS-B')
        """
        self.calc_laplace(loghyp, f=f0)
        return _handle().gpc_evidence_grad()

    def predict(self, loghyp, z):
        """Latent mean, latent variance and class probability at the test inputs z (R&W Alg. 3.2).

        The factorisation lives in the device work space of the last ``calc_laplace``; it is
        refreshed here (warm-started at the stored mode when the hyper-parameters are unchanged) so
        that interleaved calls on other objects cannot leave stale state behind.
        """
        warm = self._f_hat if (self._loghyp is not None and np.array_equal(self._loghyp, np.asarray(loghyp, dtype=float))) else None
        self.calc_laplace(loghyp, f=warm)
        z = np.asarray(z, dtype=float)
        return _handle().gpc_predict(z.reshape(len(z), -1))
