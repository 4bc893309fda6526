"""CPU checks of the oracle for the hyper-parameter gradient of the preference Laplace evidence
(oracle/gppref_grad_oracle.py: laplace_evidence_grad, probit_terms), which the device gradient is tested against."""
import mpmath
import numpy as np
import pytest

from oracle import gppref_grad_oracle as O
from oracle.gppref_oracle import laplace_evidence


def make_data(n, P, D, seed, repeat=False, isolated=False):
    rng = np.random.default_rng(seed)
    x = rng.random((n, D))
    m = n - 1 if isolated else n                  # item n - 1 is in no pair: its row of W is zero
    uvi = rng.integers(0, m, (P, 2))
    bad = uvi[:, 0] == uvi[:, 1]
    uvi[bad, 1] = (uvi[bad, 0] + 1) % m
    if repeat:                                    # the same comparisons several times, in both orientations
        uvi = np.concatenate([uvi, uvi[:P // 3], uvi[:P // 5, ::-1]])
    lat = np.sin(4 * x.sum(1))
    y = np.where(lat[uvi[:, 1]] - lat[uvi[:, 0]] + 0.3 * rng.standard_normal(len(uvi)) > 0, 1.0, -1.0)
    return x, uvi, y


def evidence_at(th, x, uvi, y):
    sigma = np.exp(th[-1])
    f = O.laplace_mode(x, uvi, y, th, sigma, tol=1e-13)
    return laplace_evidence(x, uvi, y, th, f, sigma)


CASES = [(1, 1.0, False, False), (2, 1.0, False, False), (3, 1.0, False, False),
         (1, 0.02, False, False), (2, 0.02, False, False), (3, 0.02, False, False),
         (2, 0.4, True, False), (2, 0.4, False, True)]


@pytest.mark.parametrize("D,sigma,repeat,isolated", CASES)
def test_oracle_gradient_matches_central_differences(D, sigma, repeat, isolated):
    x, uvi, y = make_data(40, 150, D, seed=D, repeat=repeat, isolated=isolated)
    th = np.log([0.3] * D + [1.2, sigma])
    f = O.laplace_mode(x, uvi, y, th, sigma, tol=1e-13)
    ev, g = O.laplace_evidence_grad(x, uvi, y, th, f, sigma)
    assert ev == laplace_evidence(x, uvi, y, th, f, sigma)
    # 5-point stencil.  Every evaluation is a fresh mode with cond(K) ~ 1e7, which wants a wide step; at sigma = 0.02
    # the evidence curves sharply in the length-scales, which wants a narrow one
    hh = 3e-3 if sigma > 0.1 else 1e-4
    fd = np.empty(len(th))
    for j in range(len(th)):
        e = np.zeros(len(th))
        e[j] = hh
        fd[j] = (-evidence_at(th + 2 * e, x, uvi, y) + 8 * evidence_at(th + e, x, uvi, y)
                 - 8 * evidence_at(th - e, x, uvi, y) + evidence_at(th - 2 * e, x, uvi, y)) / (12 * hh)
    assert np.abs(g - fd).max() <= 1e-6 * np.abs(g).max(), (g, fd)


def test_probit_terms_match_mpmath():
    mpmath.mp.dps = 50
    z = np.concatenate([np.linspace(-40, 40, 1601), [-3.0, np.nextafter(-3.0, 0), -5.0, -30.0]])
    r, w, r2 = O.probit_terms(z)
    ref = np.empty((len(z), 3))
    for i, zi in enumerate(z):
        t = mpmath.mpf(zi)
        rr = mpmath.npdf(t) / mpmath.ncdf(t)
        ref[i] = [float(rr), float(rr * (t + rr)), float(rr * ((t + rr) * (t + 2 * rr) - 1))]
    # r, w and r2 of z > 37.5 are below DBL_MIN (z > 38.5: 0 in float64): there only an absolute bound applies
    for got, want in zip((r, w, r2), ref.T):
        assert np.all(np.abs(got - want) <= 1e-10 * np.abs(want) + 1e-300)
    grid = z[:1601] <= 37                          # w = -(log Phi)'' falls monotonically, r2 = -w' > 0
    assert np.all(r2[:1601][grid] > 0) and np.all(np.diff(w[:1601][grid]) <= 0)
