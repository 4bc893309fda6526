"""The slice of GPy that ``GP_parameter_fit.py`` uses, on the B200 path.

The reference's fourth script does its regression through GPy (un-vendored, un-pinned):
``GPy.kern.RBF(input_dim=2, variance=10., lengthscale=20.)``, ``GPy.models.GPRegression(X, Y, kernel)``,
``gpm.optimize(messages=True)``, ``gpm.optimize_restarts(num_restarts=10)``, ``gpm.set_XY(...)`` and
``gpm.predict(Xfull)`` (GP_parameter_fit.py:30-33,52,62).  This module provides those names with the same call
signatures and return shapes, so the numeric part of that script runs with

    import gptest_b200.gpy_compat as GPy

PARITY UNPINNED: GPy is not in /root/reference and no version is pinned; semantics are restated from GPy's
documentation (zero mean, Gaussian noise variance 1.0 by default, ``predict`` returns (M,1) mean and (M,1)
variance INCLUDING the noise variance, positive parameters optimised in an unconstrained space, restarts drawn
from a standard normal in that space).  What is checked (tests/test_gpu_gpy_compat.py) is the arithmetic: log
likelihood, gradients and predictions against the CPU oracle of the same kernel.

Every likelihood / gradient / prediction is a call into libgpb200 (value + gradient: factorisation, identity
sweep, U U^T and the fused trace kernel); the L-BFGS iterations themselves are host code (scipy), as they are in
GPy.  ``optimize_restarts`` advances all restarts in lock step so that each iteration is ONE batched device call
(gptest_b200.sweep.multistart_fit) instead of GPy's sequential loop.
"""
import numpy as np

from . import _lib
from . import sweep as _sweep


class _Kern(object):
    pass


class RBF(_Kern):
    """``GPy.kern.RBF``: k(x,x') = variance * exp(-0.5 * |x-x'|^2 / lengthscale^2) (per-dimension with ARD=True)."""

    def __init__(self, input_dim, variance=1., lengthscale=None, ARD=False, active_dims=None, name='rbf'):
        self.input_dim = int(input_dim)
        self.ARD = bool(ARD)
        self.variance = float(variance)
        n = self.input_dim if self.ARD else 1
        if lengthscale is None:
            lengthscale = np.ones(n)
        self.lengthscale = np.broadcast_to(np.asarray(lengthscale, dtype=float).reshape(-1), (n,)).copy()
        self.name = name

    def _ell(self):
        return np.broadcast_to(np.asarray(self.lengthscale, dtype=float).reshape(-1), (self.input_dim,)) \
            if not self.ARD else np.asarray(self.lengthscale, dtype=float).reshape(-1)

    def K(self, X, X2=None):
        h = _lib.default_handle()
        X = np.asarray(X, dtype=float).reshape(len(X), -1)
        h.set_train(X)
        kh = np.concatenate([self._ell(), [self.variance, 0.0]])
        if X2 is None:
            return h.kxx(kh, flags=1)
        return h.kxz(kh, np.asarray(X2, dtype=float).reshape(len(X2), -1))


class kern(object):          # noqa: N801 - GPy spells it ``GPy.kern.RBF``
    RBF = RBF


class _Gaussian(object):
    def __init__(self, variance=1.0):
        self.variance = float(variance)


class GPRegression(object):
    """``GPy.models.GPRegression(X, Y, kernel=None, noise_var=1.)`` - exact GP regression, zero mean."""

    def __init__(self, X, Y, kernel=None, Y_metadata=None, normalizer=None, noise_var=1.0, mean_function=None):
        self.kern = kernel if kernel is not None else RBF(np.asarray(X).shape[1])
        self.likelihood = _Gaussian(noise_var)
        self.Gaussian_noise = self.likelihood
        self.set_XY(X, Y)

    # ---- data ----------------------------------------------------------------------------------------
    def set_XY(self, X=None, Y=None):
        """GP_parameter_fit.py:62 - replace the training set (the hyper-parameters stay)."""
        if X is not None:
            self.X = np.asarray(X, dtype=float).reshape(len(X), -1)
        if Y is not None:
            self.Y = np.asarray(Y, dtype=float).reshape(len(Y), -1)
        assert self.X.shape[0] == self.Y.shape[0] and self.Y.shape[1] == 1

    def _sync_factor(self):
        """Bring the factor stored on the device (gpb_gpr_grow_*) in line with (X, Y, parameters).

        The script's replay loop (GP_parameter_fit.py:61-63) calls set_XY with ever longer prefixes and predicts
        after each: when the data only GREW and the parameters did not change, only the new rows are appended
        to the factor (O(n^2 m) instead of a refit); otherwise it is rebuilt.  Repeated predictions reuse it."""
        h = _lib.default_handle()
        n, d = self.X.shape
        key = self._theta().tobytes()
        st = getattr(h, '_grow_state', None)
        y = self.Y[:, 0]
        reuse = (st is not None and st['owner'] is self and st['key'] == key and st['n'] <= n <= st['cap']
                 and h.grow_size() == st['n']
                 and np.array_equal(st['X'][:st['n']], self.X[:st['n']]) and np.array_equal(st['y'][:st['n']], y[:st['n']]))
        if not reuse:
            cap = max(1024, min(2 * n, n + 8192))
            h.grow_begin(_sweep.natural_params(self._full_log_hyp(self._theta()))[0], d, cap)
            st = {'owner': self, 'key': key, 'n': 0, 'cap': cap}
            h._grow_state = st
        if st['n'] < n:
            st['n'] = -1                                    # a failing append leaves no reusable state
            self._last_nlml = h.grow_append(self.X[h.grow_size():n], y[h.grow_size():n])
            st['n'] = n
        st['X'], st['y'] = self.X.copy(), y.copy()
        return h

    # ---- parameters: [log lengthscale (1 or D), log sigma_f, log sigma_n] ------------------------------
    def _theta(self):
        return np.concatenate([np.log(np.asarray(self.kern.lengthscale, dtype=float).reshape(-1)),
                               [0.5 * np.log(self.kern.variance), 0.5 * np.log(self.likelihood.variance)]])

    def _set_theta(self, th):
        nl = len(th) - 2
        self.kern.lengthscale = np.exp(th[:nl])
        self.kern.variance = float(np.exp(2 * th[nl]))
        self.likelihood.variance = float(np.exp(2 * th[nl + 1]))

    def _full_log_hyp(self, th):
        """expand to the library's layout [log l_1..l_D, log sf, log sn] (GPr.py:93-97)"""
        d = self.X.shape[1]
        nl = len(th) - 2
        ell = th[:nl] if nl == d else np.repeat(th[:1], d)
        return np.concatenate([ell, th[nl:]])

    def _fold_grad(self, g, nl):
        d = self.X.shape[1]
        return g if nl == d else np.concatenate([[np.sum(g[:d])], g[d:]])

    @property
    def param_array(self):
        return np.concatenate([[self.kern.variance], np.asarray(self.kern.lengthscale).reshape(-1), [self.likelihood.variance]])

    # ---- likelihood ------------------------------------------------------------------------------------
    def _nlml_and_grad(self, th):
        h = _lib.default_handle()
        h.set_train(self.X, self.Y[:, 0])
        lh = self._full_log_hyp(th)
        v, g = h.gpr_nlml(_sweep.natural_params(lh)[0], want_grad=True)
        return v, self._fold_grad(g, len(th) - 2)

    def log_likelihood(self):
        h = _lib.default_handle()
        h.set_train(self.X, self.Y[:, 0])
        return -h.gpr_nlml(_sweep.natural_params(self._full_log_hyp(self._theta()))[0])

    def objective_function(self):
        return -self.log_likelihood()

    # ---- optimisation -----------------------------------------------------------------------------------
    def optimize(self, optimizer=None, messages=False, max_iters=1000, **kwargs):
        """GP_parameter_fit.py:32 - L-BFGS on the negative log marginal likelihood with device gradients."""
        import scipy.optimize as op

        def fun(th):
            try:
                return self._nlml_and_grad(th)
            except np.linalg.LinAlgError:
                return 1e25, np.zeros_like(th)

        res = op.minimize(fun, self._theta(), jac=True, method='L-BFGS-B',
                          options={'maxiter': int(max_iters), 'ftol': 1e-12, 'gtol': 1e-8})
        self._set_theta(res.x)
        if messages:
            print('optimize: %d iterations, objective %.6f' % (res.nit, res.fun))
        self.optimization_runs = getattr(self, 'optimization_runs', []) + [res]
        return res

    def optimize_restarts(self, num_restarts=10, robust=False, verbose=False, parallel=False, num_processes=None,
                          n_iter=60, seed=0, **kwargs):
        """GP_parameter_fit.py:33 - restarts from N(0,1) draws in the unconstrained space, best one kept
        (the current parameters compete as start 0).  All restarts advance in lock step: one batched
        value+gradient call per iteration (sharded over the ranks of an initialised process group)."""
        th0 = self._theta()
        nl = len(th0) - 2

        def evaluate(X, y, log_hyp, want_grad):
            h = _lib.default_handle()
            h.set_train(X, y)
            full = np.array([self._full_log_hyp(l) for l in log_hyp])
            kh = _sweep.natural_params(full)
            vals, grads, info = h.gpr_nlml_batched(kh, want_grad=True)
            vals = np.where(info == 0, vals, np.inf)
            return vals, np.array([self._fold_grad(g, nl) for g in grads])

        best, fbest, xs, fs = _sweep.multistart_fit(self.X, self.Y[:, 0], th0, n_restarts=num_restarts,
                                                    n_iter=n_iter, seed=seed, evaluate=evaluate)
        if fbest <= -self.log_likelihood() + 1e-12:
            self._set_theta(best)
        if verbose:
            for i, f in enumerate(fs):
                print('Optimization restart %d/%d, f = %s' % (i + 1, len(fs), f))
        self.restart_objectives = fs
        return self

    # ---- prediction --------------------------------------------------------------------------------------
    def predict(self, Xnew, full_cov=False, Y_metadata=None, kern=None, likelihood=None, include_likelihood=True):
        """GP_parameter_fit.py:52 - (mean (M,1), variance (M,1)); the variance includes the noise variance.
        full_cov=True: the variance is the (M,M) joint covariance (noise variance on its diagonal), from a refit."""
        Xnew = np.asarray(Xnew, dtype=float).reshape(len(Xnew), -1)
        if full_cov:
            fz, cov = self._refit_handle().gpr_predict_full(self._khyp(), Xnew, noisy=include_likelihood)
            return fz.reshape(-1, 1), cov
        h = self._sync_factor()
        fz, cov = h.grow_predict(Xnew)
        if include_likelihood:
            cov = cov + self.likelihood.variance
        return fz.reshape(-1, 1), cov.reshape(-1, 1)

    def predict_noiseless(self, Xnew, full_cov=False, **kwargs):
        return self.predict(Xnew, full_cov=full_cov, include_likelihood=False)

    def posterior_samples_f(self, X, size=10, seed=None, **kwargs):
        """Joint draws of the latent f at X: (N, 1, size).  Without seed= the seed comes from np.random, so
        np.random.seed makes the draws reproducible."""
        return self._samples(X, size, seed, noisy=False)

    def posterior_samples(self, X, size=10, seed=None, **kwargs):
        """Joint draws of noisy observations at X (the noise variance on the diagonal of the covariance): (N, 1, size)."""
        return self._samples(X, size, seed, noisy=True)

    def _samples(self, X, size, seed, noisy):
        if seed is None:
            seed = int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
        X = np.asarray(X, dtype=float).reshape(len(X), -1)
        s, _ = self._refit_handle().gpr_sample(self._khyp(), X, int(size), seed=seed, noisy=noisy)
        return s.T[:, None, :]

    def _refit_handle(self):
        h = _lib.default_handle()
        h.set_train(self.X, self.Y[:, 0])
        return h

    def _khyp(self):
        return _sweep.natural_params(self._full_log_hyp(self._theta()))[0]

    def __str__(self):
        return ('GP_regression: objective %.6f\n  rbf.variance %s\n  rbf.lengthscale %s\n  Gaussian_noise.variance %s'
                % (self.objective_function(), self.kern.variance, np.asarray(self.kern.lengthscale), self.likelihood.variance))


class models(object):        # noqa: N801 - GPy spells it ``GPy.models.GPRegression``
    GPRegression = GPRegression
