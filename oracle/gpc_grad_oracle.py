"""CPU oracle for the hyper-parameter gradient of the classification Laplace evidence (TEST INFRASTRUCTURE - not
product code): the checker of ``gpb_gpc_evidence_grad``.

A dense numpy restatement of the formulas in DESIGN.md section 4.3 (R&W Algorithm 5.1), built on ``gpc_oracle``
(the likelihood terms and the evidence of ``calc_laplace``, R&W eq. 3.32).  Parity is unpinned by construction: the
reference's ``GPc.py`` does not parse and has no arithmetic at all, let alone a gradient.
"""
import numpy as np
from scipy.linalg import solve_triangular

from .gpc_oracle import logit_terms, preprocess_labels, probit_terms
from .gppref_grad_oracle import probit_terms as probit_ratio_terms
from .gppref_oracle import rbf_ard_K


def third_derivative(y, f, link='probit'):
    """d^3 log p(y|f) / df^3 for an array f.

    Probit, p = Phi(y f): y r''(y f) with r'' = -w' of the preference oracle (tail-safe below y f = -3).
    Logit: -pi (1 - pi)(1 - 2 pi), pi = 1 / (1 + exp(-f)), the pi the fit's W = pi (1 - pi) is made of."""
    y = np.asarray(y, dtype=float)
    f = np.asarray(f, dtype=float)
    if link == 'Logit':
        pi = 1.0 / (1.0 + np.exp(-f))
        return -(pi * (1.0 - pi)) * (1.0 - 2.0 * pi)
    return y * probit_ratio_terms(y * f)[2]


def laplace_evidence_grad(x, y, loghyp, f, link='probit', eps=1e-6):
    """(lml, d lml / d[log l_1..log l_D, log sf]) at the mode f, with the jitter eps held fixed.

    K = K_se + eps I, a = K^-1 f (through B, see below), W = -d2 log p, B = I + W^1/2 K W^1/2, lml = -a'f/2 + sum log p - sum log diag chol(B),
    R = W^1/2 B^-1 W^1/2, Sigma_ii = K_ii - |column i of L_B^-1 W^1/2 K|^2, s2 = +1/2 Sigma_ii d3_i,
    t = s2 - R K s2, b = a/2 + t, M = R - a b' - b a',  d lml / d theta_j = -1/2 tr(M dK/dtheta_j)
    (dK/dlog sf = 2 sf2 k_SE).  Exact only at a stationary point of log p(y|f) - f'K^-1 f / 2."""
    x = np.asarray(x, dtype=float).reshape(len(x), -1)
    y = preprocess_labels(y)
    f = np.asarray(f, dtype=float).reshape(-1)
    n, D = x.shape
    ell = np.exp(loghyp[:D])
    sf2 = np.exp(loghyp[D]) ** 2
    Kse = rbf_ard_K(x, ell, sf2)
    K = Kse + eps * np.eye(n)
    terms = logit_terms if link == 'Logit' else probit_terms
    lp, g, W = terms(y, f)
    sW = np.sqrt(W)
    L = np.linalg.cholesky(np.eye(n) + sW[:, None] * K * sW[None, :])
    # a = K^-1 f at the mode, formed as R&W Alg. 3.1 line 7 does (one Newton step from f, through B only): K is
    # as ill-conditioned as the jitter lets it be, B is not
    bv = W * f + g
    a = bv - sW * solve_triangular(L, solve_triangular(L, sW * (K @ bv), lower=True), lower=True, trans='T')
    lml = -0.5 * a @ f + np.sum(lp) - np.sum(np.log(np.diag(L)))
    Li = solve_triangular(L, np.eye(n), lower=True)
    R = sW[:, None] * (Li.T @ Li) * sW[None, :]
    V = Li @ (sW[:, None] * K)
    s2 = 0.5 * (np.diag(K) - np.sum(V * V, 0)) * third_derivative(y, f, link)
    b = 0.5 * a + s2 - R @ (K @ s2)
    M = R - np.outer(a, b) - np.outer(b, a)
    xs = x / ell
    grad = [-0.5 * np.sum(M * Kse * (xs[:, j, None] - xs[None, :, j]) ** 2) for j in range(D)]
    grad.append(-0.5 * np.sum(M * 2.0 * Kse))
    return lml, np.array(grad)
