"""CPU checks of the oracle for the hyper-parameter gradient of the classification Laplace evidence
(oracle/gpc_grad_oracle.py: laplace_evidence_grad, third_derivative), which the device gradient is tested against."""
import mpmath
import numpy as np
import pytest

from oracle import gpc_oracle
from oracle import gpc_grad_oracle as O


def make_data(n, D, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((n, D))
    y = np.where(np.sin(6 * x[:, 0]) + 0.3 * rng.standard_normal(n) > 0, 1.0, -1.0)
    return x, y


def make_saturated():
    """One label against 1499 others in a tight 1-D cluster: at the mode y f < -3 for that item, where the probit
    r'' comes from the continued fraction (fewer items do not get there: the item's pull grows like -y f, the
    others' like N(f)/Phi(f))."""
    rng = np.random.default_rng(4)
    x = 0.05 * rng.random((1500, 1))
    y = np.ones(1500)
    y[0] = -1.0
    return x, y, np.log([1.0, 3.0])


def fit(x, y, th, link):
    f, lml, st = gpc_oracle.calc_laplace(x, y, th, link=link, delta_f=1e-12, max_iter=200, return_state=True)
    assert st['trace'][-1][0] <= 1e-12                # converged: the formula holds at a stationary point only
    return f, lml, st['eps']


def central_differences(x, y, th, link, step):
    eps_seen = set()

    def lml_at(t):
        _, lml, eps = fit(x, y, t, link)
        eps_seen.add(eps)
        return lml

    fd = np.empty(len(th))
    for j in range(len(th)):
        e = np.zeros(len(th))
        e[j] = step
        fd[j] = (-lml_at(th + 2 * e) + 8 * lml_at(th + e) - 8 * lml_at(th - e) + lml_at(th - 2 * e)) / (12 * step)
    return fd, eps_seen


@pytest.mark.parametrize("D,link", [(1, 'probit'), (2, 'probit'), (3, 'probit'), (1, 'Logit'), (2, 'Logit'),
                                    (3, 'Logit')])
def test_oracle_gradient_matches_central_differences(D, link):
    x, y = make_data(100, D, seed=D)
    th = np.log([0.3] * D + [2.0])
    f, lml, eps = fit(x, y, th, link)
    ev, g = O.laplace_evidence_grad(x, y, th, f, link=link, eps=eps)
    assert abs(ev - lml) <= 1e-10 * abs(lml)           # a = K^-1 f here, the Newton iterate in calc_laplace
    fd, eps_seen = central_differences(x, y, th, link, step=1e-3)
    assert eps_seen == {eps}                           # the gradient holds the jitter fixed: so must the stencil
    assert np.abs(g - fd).max() <= 1e-6 * np.abs(g).max(), (g, fd)


def test_oracle_gradient_with_saturated_items():
    x, y, th = make_saturated()
    f, lml, eps = fit(x, y, th, 'probit')
    assert (y * f).min() < -3
    ev, g = O.laplace_evidence_grad(x, y, th, f, link='probit', eps=eps)
    fd, eps_seen = central_differences(x, y, th, 'probit', step=1e-3)
    assert eps_seen == {eps}
    assert np.abs(g - fd).max() <= 1e-6 * np.abs(g).max(), (g, fd)


def test_logit_third_derivative_matches_mpmath():
    mpmath.mp.dps = 50
    f = np.linspace(-30, 30, 1201)
    got = O.third_derivative(np.ones_like(f), f, link='Logit')
    assert np.array_equal(got, O.third_derivative(-np.ones_like(f), f, link='Logit'))    # independent of y
    ref = np.array([float(mpmath.diff(lambda t: -mpmath.log1p(mpmath.exp(-t)), mpmath.mpf(v), 3)) for v in f])
    # 1 - pi is formed as in the fit's W = pi (1 - pi), so it cancels for f >> 0: the relative error grows like
    # u / (1 - pi) (1e-10 at f = 14); 1 - 2 pi cancels near f = 0, an absolute u / 4.  Both stay at the rounding of
    # d3's own scale (max 0.096).
    pi = 1.0 / (1.0 + np.exp(-f))
    assert np.all(np.abs(got - ref) <= 2e-15 * np.abs(ref) / (1.0 - pi) + 5e-17)
    assert np.abs(got - ref).max() <= 1e-15
