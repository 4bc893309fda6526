"""Device gradient of the classification Laplace evidence (gpb_gpc_evidence_grad) against the dense oracle
(oracle/gpc_grad_oracle.py: laplace_evidence_grad) at the device's mode and jitter, against central differences of
the device lml, and through the GPc drop-in with an off-the-shelf quasi-Newton optimiser."""
import numpy as np
import pytest
from scipy.special import ndtr

from bench_configs import make_c3
from oracle import gpc_grad_oracle, gpc_oracle
from oracle.gppref_oracle import rbf_ard_K
from tests.test_gpc_evidence_grad import make_saturated

pytestmark = pytest.mark.gpu
LINK = {'probit': 0, 'Logit': 1}


def gpc_khyp(loghyp, d):
    return np.concatenate([np.exp(loghyp[:d]), [np.exp(loghyp[d]) ** 2]])


def make_gpc(n, D, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((n, D))
    w = rng.standard_normal(D)
    lat = np.sin(2 * np.pi * x @ w / np.abs(w).sum() + np.pi / 4) + 0.2
    y = np.where(rng.random(n) < ndtr(lat), 1.0, -1.0)
    return x, y


def fit(handle, x, y, lh, link, delta_f=1e-10, max_iter=200):
    handle.set_train(x)
    f, lml, iters, trace, jit = handle.gpc_laplace(y, gpc_khyp(lh, x.shape[1]), link=LINK[link], delta_f=delta_f,
                                                   max_iter=max_iter)
    return f, lml, jit


def check_against_oracle(handle, x, y, lh, link, tol_lml=1e-8, tol_grad=1e-8):
    f, lml, jit = fit(handle, x, y, lh, link)
    ev, g = handle.gpc_evidence_grad()
    assert ev == lml                                # the value gpc_laplace returned, bit for bit
    rev, rg = gpc_grad_oracle.laplace_evidence_grad(x, y, lh, f, link=link, eps=jit)
    lml_err = abs(ev - rev) / abs(rev)
    grad_err = np.abs(g - rg).max() / np.abs(rg).max()
    assert lml_err <= tol_lml, (ev, rev)
    assert grad_err <= tol_grad, (g, rg)
    return f, jit, lml_err, grad_err


@pytest.mark.parametrize("n,D,link,ls", [(60, 1, 'probit', 0.4), (60, 2, 'Logit', 0.4), (300, 3, 'probit', 0.5),
                                         (300, 3, 'Logit', 0.5), (333, 2, 'probit', 0.3), (333, 2, 'Logit', 0.3),
                                         (640, 6, 'probit', 0.8), (640, 6, 'Logit', 0.8)])
def test_evidence_grad_matches_oracle(handle, n, D, link, ls):
    x, y = make_gpc(n, D, seed=n + D)
    check_against_oracle(handle, x, y, np.log([ls] * D + [1.5]), link)


def test_evidence_grad_with_saturated_items(handle):
    """One label against 1499 in a tight cluster: y f < -3 at the mode, where r'' comes from the continued fraction."""
    x, y, lh = make_saturated()
    f, jit, lml_err, grad_err = check_against_oracle(handle, x, y, lh, 'probit')
    print('saturated: min y f %.3f  lml rel %.2e  grad rel %.2e' % ((y * f).min(), lml_err, grad_err))
    assert (y * f).min() < -3


@pytest.mark.parametrize("link", ['probit', 'Logit'])
def test_evidence_grad_ill_conditioned_1d(handle, link):
    """Dense 1-D inputs: cond(K + eps I) > 1e8 at the 1e-6 jitter, held to 1e-6 of max|grad| (DESIGN.md section 9
    has the measured figure)."""
    x, y = make_gpc(600, 1, seed=11)
    lh = np.log([0.5, 1.0])
    f, jit, lml_err, grad_err = check_against_oracle(handle, x, y, lh, link, tol_lml=1e-8, tol_grad=1e-6)
    cond = np.linalg.cond(rbf_ard_K(x, np.exp(lh[:1]), np.exp(lh[1]) ** 2) + jit * np.eye(len(x)))
    print('ill-conditioned 1-D %s: cond %.2e  jitter %g  lml rel %.2e  grad rel %.2e' % (link, cond, jit, lml_err, grad_err))
    assert jit == 1e-6 and cond > 1e8


def central_differences(handle, x, y, lh, link, step):
    jits = set()

    def lml_at(t):
        _, lml, jit = fit(handle, x, y, t, link)
        jits.add(jit)
        return lml

    fd = np.empty(len(lh))
    for j in range(len(lh)):
        e = np.zeros(len(lh))
        e[j] = step
        fd[j] = (-lml_at(lh + 2 * e) + 8 * lml_at(lh + e) - 8 * lml_at(lh - e) + lml_at(lh - 2 * e)) / (12 * step)
    return fd, jits


@pytest.mark.parametrize("size,link", [('n300', 'probit'), ('n300', 'Logit'), ('c3', 'probit')])
def test_evidence_grad_matches_central_differences(handle, size, link):
    if size == 'c3':
        x, y, _, lh = make_c3()
    else:
        x, y = make_gpc(300, 3, seed=5)
        lh = np.log([0.4, 0.4, 0.4, 1.5])
    _, _, jit = fit(handle, x, y, lh, link)
    ev, g = handle.gpc_evidence_grad()
    fd, jits = central_differences(handle, x, y, lh, link, step=1e-3)
    assert jits == {jit}                            # the gradient holds the jitter fixed: so must the stencil
    print(size, link, 'grad', g, 'fd', fd, 'rel %.2e' % (np.abs(g - fd).max() / np.abs(g).max()))
    assert np.abs(g - fd).max() <= 1e-6 * np.abs(g).max(), (g, fd)


def test_evidence_grad_is_deterministic_and_keeps_the_state(handle):
    x, y = make_gpc(300, 3, seed=9)
    lh = np.log([0.4, 0.4, 0.4, 1.5])
    _, lml, _ = fit(handle, x, y, lh, 'probit')
    z = np.random.default_rng(3).random((70, 3))
    p0 = handle.gpc_predict(z)
    ev1, g1 = handle.gpc_evidence_grad()
    p1 = handle.gpc_predict(z)                      # the factor of B is rebuilt: the same bits
    ev2, g2 = handle.gpc_evidence_grad()
    ev3, g3 = handle.gpc_evidence_grad()            # the factor overwritten by the previous call is rebuilt first
    p2 = handle.gpc_predict(z)
    assert ev1 == lml and ev2 == lml and ev3 == lml
    assert np.array_equal(g1, g2) and np.array_equal(g1, g3)
    for a, b, c in zip(p0, p1, p2):
        assert np.array_equal(a, b) and np.array_equal(a, c)


def test_evidence_grad_errors(handle):
    from gptest_b200 import _lib
    x, y = make_gpc(80, 2, seed=2)
    lh = np.log([0.4, 0.4, 1.5])
    h = _lib.Handle(0)
    try:
        h.set_train(x)
        with pytest.raises(_lib.GpbError, match='gpb_gpc_laplace first'):
            h.gpc_evidence_grad()
    finally:
        h.close()
    fit(handle, x, y, lh, 'probit')
    handle.gpc_evidence_grad()
    handle.kxx(np.array([0.4, 0.4, 1.0, 0.0]))      # an unrelated call invalidates the state
    with pytest.raises(_lib.GpbError, match='gpb_gpc_laplace first'):
        handle.gpc_evidence_grad()
    f, lml, iters, trace, jit = handle.gpc_laplace(y, gpc_khyp(lh, 2), link=0, delta_f=1e-12, max_iter=2)
    assert iters == 2 and trace[-1, 0] > 1e-12
    z = x[:7]
    p0 = handle.gpc_predict(z)
    with pytest.raises(_lib.GpbError, match='converged mode'):
        handle.gpc_evidence_grad()
    p1 = handle.gpc_predict(z)                      # a refused call leaves the state usable
    for a, b in zip(p0, p1):
        assert np.array_equal(a, b)


def test_dropin_hyperparameter_fit_with_lbfgs(handle):
    from scipy.optimize import minimize
    from gptest_b200 import GPc
    x, y, _, lh = make_c3(n=600, d=2)
    gp = GPc.ClassifierGaussianProcess(x, y, delta_f=1e-10)

    def objective(t):
        lml, g = gp.laplace_evidence_and_grad(t, f0=gp._f_hat)
        return -lml, -g

    e0, g0 = objective(lh)
    assert g0.shape == (3,)
    res = minimize(objective, lh, jac=True, method='L-BFGS-B', options=dict(maxiter=200, ftol=1e-13, gtol=1e-9))
    e1, g1 = objective(res.x)
    print('C3 n = 600 L-BFGS-B: %d evaluations, lml %.6f -> %.6f, |grad| %.2e -> %.2e'
          % (res.nfev, -e0, -e1, np.abs(g0).max(), np.abs(g1).max()))
    assert -e1 > -e0
    assert np.abs(g1).max() < 1e-4 * np.abs(g0).max()
    mu, var, p = gp.predict(res.x, x[:5])
    assert p.shape == (5,) and np.all((p > 0) & (p < 1))
    ref = gpc_oracle.calc_laplace(x, y, lh, delta_f=1e-10)[1]
    assert abs(gp.calc_nlml(lh) + ref) <= 1e-8 * abs(ref)
