"""Drop-in replacement for the reference's ``GPr.py`` with the numerics on a B200.

Same public names, constructor signatures, attributes and return types as
/root/reference/GPr.py (cited per symbol below); ``GP_regression_demo.py:41-48`` runs
unmodified against this module.  Every dense operation (covariance assembly, Cholesky,
solves, reductions) is a CUDA kernel reached through libgpb200's C ABI - there is no numpy
fallback; only the few scalar lines that define the object attributes stay on the host.
"""
import numpy as np

from . import _lib


def _handle():
    return _lib.default_handle()


def squared_distance(A, B):
    """GPr.py:4-13 - expanded-form squared distances, (len(A), len(B)).

    The reference reshapes to one column (1-D inputs only); here 2-D inputs (N,D), (M,D) are
    accepted as well and summed over D.
    """
    A = np.asarray(A, dtype=float)
    B = np.asarray(B, dtype=float)
    A = A.reshape(len(A), -1)
    B = B.reshape(len(B), -1)
    h = _handle()
    h.set_train(A)
    return h.sqdist(B)


class GaussianProcess(object):
    """GPr.py:16-69."""

    def __init__(self, log_hyp, mean_hyp, like_hyp, covFunName, meanFunName, likeFunName,
                 trainInput, trainTarget):
        # GPr.py:19-26: plain attribute storage
        self.log_hyp = log_hyp
        self.mean_hyp = mean_hyp
        self.like_hyp = like_hyp
        self.covFunName = covFunName
        self.meanFunName = meanFunName
        self.likeFunName = likeFunName
        self.trainInput = trainInput
        self.trainTarget = trainTarget
        # GPr.py:28-42: string dispatch, unknown names give []
        if covFunName in COVARIANCE_FUNCTIONS:        # "SE" in the reference; the Matern names are extensions
            self.covFun = COVARIANCE_FUNCTIONS[covFunName](log_hyp, trainInput)
        else:
            self.covFun = []
        if meanFunName == "zero":
            self.meanFun = MeanFunction(mean_hyp)
        else:
            self.meanFun = []
        if likeFunName == "zero":
            self.likeFun = LikelihoodFunction(like_hyp)
        else:
            self.likeFun = []

    def compute_prediction(self, testInput, full_cov=False):
        """GPr.py:45-54: (fz, cov_fz) = (Kzx K^-1 y, sf2 - diag(Kzx K^-1 Kxz)).

        The reference inverts K by LU and forms an (M,M) product; here K is factored once and
        the test rows ride along the factorisation (see csrc/chol.cu), same quantities.
        full_cov=True (not in the reference): cov_fz is the whole (M,M) matrix Kzz - Kzx K^-1 Kxz, and fz is the same.
        """
        cov = self.covFun
        h = _handle()
        h.set_train(cov.x, self.trainTarget)           # GPr.py:52 uses trainTarget as is (no mean)
        if full_cov:
            return h.gpr_predict_full(cov.khyp(), testInput, kind=cov.KIND)
        fz, cov_fz = h.gpr_predict(cov.khyp(), testInput, kind=cov.KIND)
        return fz, cov_fz

    def compute_posterior_samples(self, testInput, n_samples, seed=0):
        """Joint draws of the latent f at testInput from the posterior of compute_prediction(testInput, full_cov=True):
        (n_samples, M).  Not in the reference; the draws are a function of seed alone (csrc/posterior.cu)."""
        cov = self.covFun
        h = _handle()
        h.set_train(cov.x, self.trainTarget)
        samples, _ = h.gpr_sample(cov.khyp(), testInput, n_samples, seed=seed, kind=cov.KIND)
        return samples

    def compute_likelihood(self, hyp):
        """GPr.py:57-69: negative log marginal likelihood for ``hyp``; returns a (1,1) array."""
        covSE = self._cov_class()(hyp, self.trainInput)           # GPr.py:59 (kernel from the argument)
        m = self.meanFun.y                                        # GPr.py:61
        y = np.reshape(self.trainTarget, (len(self.trainTarget), 1))   # GPr.py:64
        h = _handle()
        h.set_train(covSE.x, (y - m).reshape(-1))
        nlml = h.gpr_nlml(covSE.khyp(), kind=covSE.KIND)
        return np.array([[nlml]])

    def compute_likelihood_and_gradient(self, hyp):
        """Value and gradient w.r.t. the log hyper-parameters (not in the reference, which uses
        Nelder-Mead; this is what GPy's L-BFGS in GP_parameter_fit.py:32-33 consumes)."""
        covSE = self._cov_class()(hyp, self.trainInput)
        m = self.meanFun.y
        y = np.reshape(self.trainTarget, (len(self.trainTarget), 1))
        h = _handle()
        h.set_train(covSE.x, (y - m).reshape(-1))
        return h.gpr_nlml(covSE.khyp(), want_grad=True, kind=covSE.KIND)

    def _cov_class(self):
        # GPr.py:59 hard-codes SquaredExponential; with one of the extension names the same kernel family as covFun
        return COVARIANCE_FUNCTIONS.get(self.covFunName, SquaredExponential)


class MeanFunction(object):
    """GPr.py:72-75."""

    def __init__(self, x):
        self.x = x
        self.y = np.zeros_like(x)


class LikelihoodFunction(object):
    """GPr.py:78-81."""

    def __init__(self, x):
        self.x = x
        self.y = np.exp(2 * x)


class CovarianceFunction(object):
    """GPr.py:84-87."""

    def __init__(self, logHyp, x):
        self.logHyp = logHyp
        self.x = x


class SquaredExponential(CovarianceFunction):
    """GPr.py:90-110."""
    KIND = 0            # radial function on the device (csrc/gpb_exp.cuh)

    def __init__(self, logHyp, x):
        CovarianceFunction.__init__(self, logHyp, x)
        self.hyp = np.exp(self.logHyp)          # GPr.py:93
        n = len(self.hyp)
        self.M = self.hyp[:n - 2]               # GPr.py:95 length scales
        self.sf2 = self.hyp[n - 2] ** 2         # GPr.py:96
        self.sn2 = self.hyp[n - 1] ** 2         # GPr.py:97

    def khyp(self):
        """[l_1..l_D, sf2, sn2]: the natural parameters handed to the C ABI."""
        return np.concatenate([np.asarray(self.M, dtype=float).reshape(-1), [self.sf2, self.sn2]])

    def _points(self, z=None):
        x = np.asarray(self.x, dtype=float)
        x = x.reshape(len(x), -1)
        d = x.shape[1]
        if len(self.M) != d:
            raise ValueError('%d length scales for %d input dimensions' % (len(self.M), d))
        if z is None:
            return x
        z = np.asarray(z, dtype=float)
        return x, z.reshape(len(z), -1)

    def compute_Kxx_matrix(self):
        """GPr.py:99-103: full symmetric sn2*I + sf2*exp(-0.5*sqdist(x/M, x/M))."""
        h = _handle()
        h.set_train(self._points())
        return h.kxx(self.khyp(), kind=self.KIND)

    def compute_Kxz_matrix(self, z):
        """GPr.py:105-110."""
        x, z = self._points(z)
        h = _handle()
        h.set_train(x)
        return h.kxz(self.khyp(), z, kind=self.KIND)


class Matern32(SquaredExponential):
    """sf2 (1 + sqrt(3) r) exp(-sqrt(3) r) + sn2 I with the ARD scaling and hyper-parameter layout of GPr.py:93-100.
    Not in the reference (its string dispatch, GPr.py:28-32, knows only "SE"): SURVEY 8f rank 4."""
    KIND = 1


class Matern52(SquaredExponential):
    """sf2 (1 + sqrt(5) r + 5 r^2 / 3) exp(-sqrt(5) r) + sn2 I; see Matern32."""
    KIND = 2


COVARIANCE_FUNCTIONS = {"SE": SquaredExponential, "Matern32": Matern32, "Matern52": Matern52}
