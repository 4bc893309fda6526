"""Drop-in replacement for the reference's ``GPpref.py`` with the numerics on a B200.

Same public names and signatures as /root/reference/GPpref.py (cited per symbol);
``GP_preference_demo.py:60,67`` and ``fmin(prefGP.calc_nlml, theta0)`` run unmodified.  The
covariance assembly, the explicit inverse, every Newton iteration (likelihood derivatives, W,
the dense solve) and the objective are CUDA kernels behind libgpb200's C ABI; the reference's
GPy dependency is gone (``RBF`` below is a two-attribute stand-in whose ``K`` is the device
kernel with GPy's RBF semantics).

The reference's behaviour is reproduced on purpose, quirks included (SURVEY section 0):
last-write-wins gradient (GPpref.py:77-78), the probit sigma that never changes because
``calc_laplace`` overwrites the method ``set_sigma`` (GPpref.py:115), and ``logdetK`` being half the
log-determinant (GPpref.py:131) halved again in ``log_marginal`` (GPpref.py:93).  The opt-in
``newton=True`` constructor flag gives the accumulated gradient (true Newton steps).
"""
import numpy as np

from . import _lib

_sqrt_2pi = np.sqrt(2 * np.pi)


def _handle():
    return _lib.default_handle()


def std_norm_pdf(x):
    """GPpref.py:7-10 (scalar helper kept on the host; the device kernels have their own)."""
    x = np.clip(x, -1e150, 1e150)
    return np.exp(-(x ** 2) / 2) / _sqrt_2pi


from .GPr import squared_distance  # noqa: E402,F401  GPpref.py:13-22 (duplicate of GPr.py:4-13): same device kernel


class SquaredExponential(object):
    """GPpref.py:25-44.  In the reference this class is dead code: its constructor stores ``length`` and
    ``logvar`` while its two methods read ``self.M``, ``self.sf2`` and ``self.sn2``, which nothing sets, so any
    call raises AttributeError.  The name is kept importable with the constructor's attributes
    (GPpref.py:27-31); the methods fail the same way.  The working kernel of this module is ``RBF`` below."""

    def __init__(self, logHyp, x):
        self.x = x
        self.hyp = np.exp(logHyp)
        xdim = self.x.shape[1]
        self.length = self.hyp[0:xdim]
        self.logvar = self.hyp[-1] ** 2

    def compute_Kxx_matrix(self):
        raise AttributeError("'SquaredExponential' object has no attribute 'M'")          # GPpref.py:34

    def compute_Kxz_matrix(self, z):
        raise AttributeError("'SquaredExponential' object has no attribute 'M'")          # GPpref.py:40


class RBF(object):
    """Stand-in for ``GPy.kern.RBF(input_dim, ARD=True)`` (GPpref.py:109): holds ``lengthscale`` and
    ``variance`` and evaluates ``K`` on the device (r^2 clipped at 0, exact zero diagonal)."""

    def __init__(self, input_dim, ARD=True):
        self.input_dim = input_dim
        self.ARD = ARD
        self.lengthscale = np.ones(input_dim)
        self.variance = 1.0

    def khyp(self):
        ls = np.broadcast_to(np.asarray(self.lengthscale, dtype=float).reshape(-1), (self.input_dim,))
        return np.concatenate([ls, [float(self.variance)]])

    def K(self, X):
        h = _handle()
        h.set_train(X)
        return h.kxx(np.concatenate([self.khyp(), [0.0]]), flags=1)


class PrefProbit(object):
    """GPpref.py:46-94."""

    def __init__(self, sigma=1.0):
        self.set_sigma(sigma)
        self.log2pi = np.log(2.0 * np.pi)

    def set_sigma(self, sigma):
        self.sigma = sigma                                         # GPpref.py:52
        self._isqrt2sig = 1.0 / (self.sigma * np.sqrt(2.0))        # GPpref.py:53
        self._i2var = self._isqrt2sig ** 2                         # GPpref.py:54

    def z_k(self, uvi, f, y):
        """GPpref.py:56-58 (an index gather; stays on the host for callers that want z itself)."""
        zc = self._isqrt2sig * (f[uvi[:, 1]] - f[uvi[:, 0]])
        return y * zc

    def I_k(self, x, uv):
        """GPpref.py:60-66 (unused by the reference as well)."""
        if x == uv[0]:
            return -1
        elif x == uv[1]:
            return 1
        else:
            return 0

    def derivatives(self, uvi, y, f, accumulate=False):
        """GPpref.py:68-88: dense W (n,n) and the gradient (n,1), computed on the device."""
        f = np.asarray(f, dtype=float)
        W, g = _handle().pref_derivatives(uvi, np.asarray(y, dtype=float), f.reshape(-1), sigma=self.sigma,
                                          grad_mode=1 if accumulate else 0)
        return W, g.reshape(-1, 1)

    def log_marginal(self, uvi, y, f, iK, logdetK):
        """GPpref.py:90-94 for caller-supplied iK / logdetK, reduced on the device (the same kernel that
        ``calc_laplace`` uses per iteration); returns a python float like the reference's ``psi.flat[0]``."""
        return _handle().pref_log_marginal(uvi, y, f, iK, float(np.asarray(logdetK).reshape(-1)[0]), sigma=self.sigma)


class PreferenceGaussianProcess(object):
    """GPpref.py:96-161."""

    def __init__(self, x_train, uvi_train, y_train, likelihood=PrefProbit, delta_f=1e-6, newton=False,
                 max_iter=10000):
        # log_hyp layout: [length_0, ..., length_d, sigma_f, sigma_probit]  (GPpref.py:99)
        self._xdim = x_train.shape[1]
        self._nx = x_train.shape[0]
        self.x_train = x_train
        self.y_train = y_train
        self.uvi_train = uvi_train
        self.delta_f = delta_f
        self.likelihood = likelihood()
        self.kern = RBF(self._xdim, ARD=True)
        self.newton = newton            # not in the reference: accumulate the gradient (true Newton)
        self.max_iter = max_iter        # the reference loops without a cap (GPpref.py:140)
        self.trace = None               # per-iteration (f_error, lml): what the reference prints (GPpref.py:154)
        self.n_iter = 0
        self.jitter = None
        self.f_mode = None              # mode of the last laplace_evidence_and_grad fit (not in the reference)

    def calc_laplace(self, loghyp, f=None):
        """GPpref.py:112-157: returns (f (n,1), lml)."""
        self.kern.lengthscale = np.exp(loghyp[0:self._xdim])              # GPpref.py:113
        self.kern.variance = (np.exp(loghyp[self._xdim])) ** 2            # GPpref.py:114
        self.likelihood.set_sigma = np.exp(loghyp[-1])                    # GPpref.py:115 (sic: sigma unchanged)
        h = _handle()
        h.set_train(self.x_train)
        f0 = None if f is None else np.asarray(f, dtype=float).reshape(-1)
        fv, lml, iters, trace, jitter = h.pref_laplace(
            self.uvi_train, np.asarray(self.y_train, dtype=float).reshape(-1), self.kern.khyp(),
            sigma=self.likelihood.sigma, delta_f=self.delta_f, max_iter=self.max_iter,
            grad_mode=1 if self.newton else 0, f0=f0)
        self.trace, self.n_iter, self.jitter = trace, iters, jitter
        return fv.reshape(-1, 1), lml

    def calc_nlml(self, loghyp):
        """GPpref.py:159-161."""
        f, lml = self.calc_laplace(loghyp)
        return -lml

    # ---- opt-in extensions, NOT in the reference (SURVEY 8f rank 3; include/gpb200.h gpb_pref_evidence/_predict) ----
    # They use the state calc_laplace left on the device: call them right after it.
    def laplace_evidence(self):
        """R&W eq. 3.32 at the mode: sum log Phi(z) - f'K^-1 f/2 - log|I + K W|/2 (what GPpref.py:90-94 leaves out)."""
        return _handle().pref_evidence()

    def laplace_evidence_and_grad(self, loghyp, f0=None):
        """(evidence, grad) for hyper-parameter fitting: the Laplace evidence (as ``laplace_evidence``) and its exact
        gradient with respect to ``loghyp`` = [log l_1 .. log l_d, log sf, log sigma] (GPpref.py:99), at the mode of a
        fresh fit that accumulates the gradient (true Newton) and uses sigma = exp(loghyp[-1]) as the probit noise.
        The fit's jitter is held fixed in the gradient.  ``f0``: starting point of the Newton iteration, e.g. the
        mode of the previous call (``self.f_mode``).  Maximise the evidence, e.g.
        ``scipy.optimize.minimize(lambda t: tuple(-v for v in gp.laplace_evidence_and_grad(t)), x0, jac=True)``.

        ``calc_laplace`` / ``calc_nlml`` are unaffected (they keep the reference's sigma and gradient), but the device
        state is this fit's: ``laplace_evidence``, ``predict_latent`` and ``predict_preference`` called after this
        method use its mode, its hyper-parameters and this sigma."""
        loghyp = np.asarray(loghyp, dtype=float).reshape(-1)
        self.kern.lengthscale = np.exp(loghyp[0:self._xdim])
        self.kern.variance = (np.exp(loghyp[self._xdim])) ** 2
        h = _handle()
        h.set_train(self.x_train)
        f0 = None if f0 is None else np.asarray(f0, dtype=float).reshape(-1)
        fv, lml, iters, trace, jitter = h.pref_laplace(
            self.uvi_train, np.asarray(self.y_train, dtype=float).reshape(-1), self.kern.khyp(),
            sigma=float(np.exp(loghyp[-1])), delta_f=self.delta_f, max_iter=self.max_iter, grad_mode=1, f0=f0)
        self.trace, self.n_iter, self.jitter = trace, iters, jitter
        self.f_mode = fv
        return h.pref_evidence_grad()

    def predict_latent(self, x_test):
        """Posterior mean and variance of the latent utility at new items: ((m,), (m,))."""
        return _handle().pref_predict(x_test)

    def predict_preference(self, x_a, x_b):
        """Posterior of f(x_b) - f(x_a) and P(x_b preferred to x_a) = Phi(mean / sqrt(2 sigma^2 + var))."""
        return _handle().pref_predict(x_a, x_b)
