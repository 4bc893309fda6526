"""Generate tests/golden/* by RUNNING THE REFERENCE in this container, and check the oracle.

Run here (the dev container), never on the GPU box: it reads /root/reference, which does
not travel.  Usage:  python -m oracle.make_golden

  * GPr: /root/reference/GPr.py is imported unmodified.  KAT-1 = the data of
    GP_regression_demo.py:6-38 (seed 0, 20 points, log_hyp = log([1,1,0.1]), 100 test
    points); KAT-2 = 1024 points of sin(6x) + noise (SURVEY section 4).  The oracle
    restatement (oracle/gpr_oracle.py) must reproduce every value bit-for-bit.
  * GPpref: /root/reference/GPpref.py is Python 2 and imports GPy.  Its source is read, the
    two ``print`` statements (GPpref.py:135,154) are commented out IN MEMORY, a stub ``GPy``
    module providing ``kern.RBF`` (the oracle's restatement of GPy's RBF - the un-pinnable
    part) is injected, and the module is exec'd.  Everything else that runs - PrefProbit,
    the jitter loop, the Laplace loop - is the reference's own code.  KAT-3 = the demo data
    (GP_preference_demo.py:7-12,39-44); KAT-4 = random pairs with repeated items, which
    exercises the last-write-wins gradient.
"""
import json
import os
import re
import sys
import types

import numpy as np

REF = '/root/reference'
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))   # also runnable as a plain script
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')


def load_reference_gpr():
    sys.path.insert(0, REF)
    try:
        import GPr  # noqa: the reference module, unmodified
    finally:
        sys.path.pop(0)
    assert os.path.abspath(GPr.__file__).startswith(REF)
    return GPr


def load_reference_gppref():
    from oracle.gppref_oracle import rbf_ard_K

    class RBF:                       # stand-in for GPy.kern.RBF(input_dim, ARD=True)
        def __init__(self, input_dim, ARD=False):
            self.lengthscale = np.ones(input_dim)
            self.variance = 1.0

        def K(self, X):
            return rbf_ard_K(X, self.lengthscale, self.variance)

    gpy = types.ModuleType('GPy')
    gpy.kern = types.SimpleNamespace(RBF=RBF)
    src = open(os.path.join(REF, 'GPpref.py')).read()
    src, nsub = re.subn(r'^(\s*)print (.*)$', r'\1pass  # py2 print removed: \2', src, flags=re.M)
    assert nsub == 2, nsub
    # numpy 2 removed the np.linalg.linalg alias used at GPpref.py:133
    src = src.replace('np.linalg.linalg.LinAlgError', 'np.linalg.LinAlgError')
    mod = types.ModuleType('GPpref_reference')
    sys.modules['GPy'] = gpy
    try:
        exec(compile(src, os.path.join(REF, 'GPpref.py'), 'exec'), mod.__dict__)
    finally:
        del sys.modules['GPy']
    return mod


def demo_regression_data():
    """GP_regression_demo.py:6,9-17,27-28,32 (numeric part only)."""
    np.random.seed(0)
    c = np.array([3, 5, -9, -3, 2], float)
    x_train = np.random.random(20)
    y_train = np.polyval(c, x_train) + np.random.normal(0, 0.1, len(x_train))
    x_test = np.arange(0, 1, 0.01, float)
    return x_train, y_train, x_test


def demo_preference_data():
    """GP_preference_demo.py:7-12,15-29,39-44."""
    np.random.seed(1)
    n_train, true_sigma = 20, 0.05
    x_train = np.random.random((2 * n_train, 1))
    uvi = np.random.choice(range(2 * n_train), (n_train, 2), replace=False)
    uv = x_train[uvi][:, :, 0]
    fuv = (np.sin(uv * 2 * np.pi + np.pi / 4) + 0.2) + np.random.normal(scale=true_sigma, size=uv.shape)
    y = -1 * np.ones((fuv.shape[0], 1), dtype='int')
    y[fuv[:, 1] > fuv[:, 0]] = 1
    return x_train, uvi, y


def main():
    from oracle import gpr_oracle, gppref_oracle
    os.makedirs(OUT, exist_ok=True)
    GPr = load_reference_gpr()
    kat = {}

    # ---- KAT-1 -------------------------------------------------------------------------
    x, y, z = demo_regression_data()
    lh = np.log([1, 1, 0.1])
    gp = GPr.GaussianProcess(lh, 0, 0, "SE", "zero", "zero", x, y)
    nl = gp.compute_likelihood(lh)
    mean, var = gp.compute_prediction(z)
    K = gp.covFun.compute_Kxx_matrix()
    Kxz = gp.covFun.compute_Kxz_matrix(z)
    assert nl.shape == (1, 1)
    assert np.array_equal(K, gpr_oracle.kxx(lh, x))
    assert np.array_equal(Kxz, gpr_oracle.kxz(lh, x, z))
    assert np.array_equal(nl, gpr_oracle.nlml(lh, x, y))
    om, ov = gpr_oracle.predict(lh, x, y, z)
    assert np.array_equal(mean, om) and np.array_equal(var, ov)
    kat['kat1'] = dict(x=x.tolist(), y=y.tolist(), z=z.tolist(), log_hyp=lh.tolist(),
                       nlml=float(nl[0, 0]), K=K.tolist(), mean=mean.tolist(), var=var.tolist(),
                       Kxz_col0=Kxz[:, 0].tolist())

    # ---- KAT-1b: the demo's fmin result (optimiser-version dependent; smoke only) -------
    import scipy.optimize as op
    opt = op.fmin(gp.compute_likelihood, lh, disp=False)
    gp2 = GPr.GaussianProcess(opt, 0, 0, "SE", "zero", "zero", x, y)
    m2, v2 = gp2.compute_prediction(z)
    kat['kat1b'] = dict(opt_log_hyp=opt.tolist(), nlml=float(gp.compute_likelihood(opt)[0, 0]),
                        mean=m2.tolist(), var=v2.tolist())

    # ---- KAT-2 -------------------------------------------------------------------------
    rng = np.random.default_rng(0)
    x = rng.random(1024)
    y = np.sin(6 * x) + 0.1 * rng.standard_normal(1024)
    z = rng.random(256)
    lh = np.log([0.2, 1, 0.1])
    gp = GPr.GaussianProcess(lh, 0, 0, "SE", "zero", "zero", x, y)
    nl = gp.compute_likelihood(lh)
    mean, var = gp.compute_prediction(z)
    assert np.array_equal(nl, gpr_oracle.nlml(lh, x, y))
    om, ov = gpr_oracle.predict(lh, x, y, z)
    assert np.array_equal(mean, om) and np.array_equal(var, ov)
    kat['kat2'] = dict(recipe="rng=default_rng(0); x=rng.random(1024); y=sin(6x)+0.1*rng.standard_normal(1024); z=rng.random(256)",
                       log_hyp=lh.tolist(), nlml=float(nl[0, 0]), mean=mean.tolist(), var=var.tolist())

    # ---- KAT-2b: better conditioned 1-D case (sn = 0.3) where inv() noise is small -----
    lh = np.log([0.3, 1.0, 0.3])
    gp = GPr.GaussianProcess(lh, 0, 0, "SE", "zero", "zero", x[:512], y[:512])
    nl = gp.compute_likelihood(lh)
    mean, var = gp.compute_prediction(z)
    kat['kat2b'] = dict(recipe="first 512 points of kat2, same z", log_hyp=lh.tolist(),
                        nlml=float(nl[0, 0]), mean=mean.tolist(), var=var.tolist())
    with open(os.path.join(OUT, 'gpr_kat.json'), 'w') as fh:
        json.dump(kat, fh)

    # ---- KAT-3 / KAT-4: preference Laplace ----------------------------------------------
    ref = load_reference_gppref()
    out = {}
    x, uvi, y = demo_preference_data()
    lh = np.log([0.1, 1.0, 0.1])                      # GP_preference_demo.py:7
    gp = ref.PreferenceGaussianProcess(x, uvi, y, delta_f=1e-5)   # :12,60
    f, lml = gp.calc_laplace(lh)
    assert gp.likelihood.sigma == 1.0                 # quirk 2
    of, olml, otrace = gppref_oracle.calc_laplace(x, uvi, y, lh, delta_f=1e-5, return_trace=True)
    assert np.array_equal(f, of) and lml == olml, (np.abs(f - of).max(), lml, olml)
    W, g = gp.likelihood.derivatives(uvi, y, f)
    oW, og = gppref_oracle.ProbitPrefOracle().derivatives(uvi, y, f)
    assert np.array_equal(W, oW) and np.array_equal(g, og)
    out.update(k3_x=x, k3_uvi=uvi, k3_y=y, k3_loghyp=lh, k3_f=f, k3_lml=lml,
               k3_trace=np.array(otrace), k3_W=W, k3_g=g)

    rng = np.random.default_rng(3)
    n, P, D = 96, 400, 3
    x = rng.random((n, D))
    uvi = rng.integers(0, n, (P, 2))
    bad = uvi[:, 0] == uvi[:, 1]
    uvi[bad, 1] = (uvi[bad, 0] + 1) % n
    w = rng.standard_normal(D)
    lat = np.sin(2 * np.pi * x @ w / np.abs(w).sum() + np.pi / 4) + 0.2
    fu = lat[uvi[:, 0]] + 0.05 * rng.standard_normal(P)
    fv = lat[uvi[:, 1]] + 0.05 * rng.standard_normal(P)
    y = np.where(fv > fu, 1, -1).reshape(-1, 1)
    lh = np.log([0.5] * D + [1.0, 0.1])
    gp = ref.PreferenceGaussianProcess(x, uvi, y, delta_f=1e-6)
    f, lml = gp.calc_laplace(lh)
    of, olml, otrace = gppref_oracle.calc_laplace(x, uvi, y, lh, delta_f=1e-6, return_trace=True)
    assert np.array_equal(f, of) and lml == olml
    W, g = gp.likelihood.derivatives(uvi, y, f)
    oW, og = gppref_oracle.ProbitPrefOracle().derivatives(uvi, y, f)
    assert np.array_equal(W, oW) and np.array_equal(g, og)
    out.update(k4_x=x, k4_uvi=uvi, k4_y=y, k4_loghyp=lh, k4_f=f, k4_lml=lml,
               k4_trace=np.array(otrace), k4_g=g, k4_Wdiag=np.diag(W).copy())
    np.savez_compressed(os.path.join(OUT, 'gppref_kat.npz'), **out)
    print('golden vectors written to', OUT)
    print('kat1 nlml', kat['kat1']['nlml'], 'kat2 nlml', kat['kat2']['nlml'])
    print('kat3 iters', len(out['k3_trace']), 'lml', out['k3_lml'], '| kat4 iters', len(out['k4_trace']), 'lml', out['k4_lml'])


if __name__ == '__main__':
    from threadpoolctl import threadpool_limits
    from oracle import GOLDEN_BLAS_THREADS
    with threadpool_limits(GOLDEN_BLAS_THREADS, user_api='blas'):
        main()
