"""CPU oracle for the hyper-parameter gradient of the preference Laplace evidence (TEST INFRASTRUCTURE - not product
code): the checker of ``gpb_pref_evidence_grad``.

A dense numpy restatement of the formulas in DESIGN.md section 4.3, built on the evidence of ``gppref_oracle``
(``laplace_evidence``, R&W eq. 3.32).  Parity is unpinned by construction: the reference has no evidence and no
gradient (its hyper-optimisation, GP_preference_demo.py:66, is Nelder-Mead on ``calc_nlml``).
"""
import numpy as np
from scipy.special import ndtr

from .gppref_oracle import ProbitPrefOracle, laplace_evidence, rbf_ard_K

_SQRT_2PI = np.sqrt(2 * np.pi)

PROBIT_CF_BELOW = -3.0     # z below this: continued fraction of the Mills ratio (what the device kernel does too)
PROBIT_CF_DEPTH = 64


def probit_terms(z):
    """r = N(z)/Phi(z), w = r (z + r) = -(log Phi)'' and r2 = r ((z + r)(z + 2r) - 1) = -w' for an array z.

    Above PROBIT_CF_BELOW the closed forms are used.  Below it r z + r^2 - 1 and q = z + r cancel (r2 would lose
    ~3e-11 relative at z = -5 and 2e-5 at z = -30), so with x = -z and the continued fraction of the Mills ratio,
    c_k = k / (x + c_{k+1}):  r = x + c_1,  q = c_1,  w = r c_1,  r2 = r c_1^2 c_2 (c_3 - c_2), free of cancellation."""
    z = np.asarray(z, dtype=float)
    with np.errstate(divide='ignore', invalid='ignore', under='ignore'):
        r = np.exp(-0.5 * z * z) / _SQRT_2PI / ndtr(z)
    q = z + r
    r2 = r * (q * (z + 2.0 * r) - 1.0)
    tail = z < PROBIT_CF_BELOW
    if np.any(tail):
        x = -z[tail]
        c = np.zeros_like(x)
        cs = {}
        for k in range(PROBIT_CF_DEPTH, 0, -1):
            c = k / (x + c)
            cs[k] = c
        rt = x + cs[1]
        r[tail] = rt
        q[tail] = cs[1]
        r2[tail] = rt * cs[1] * cs[1] * cs[2] * (cs[3] - cs[2])
    return r, r * q, r2


def laplace_mode(x, uvi, y, loghyp, sigma=1.0, eps=1e-6, tol=1e-13, max_iter=200):
    """Mode of sum log Phi(z) - f'K^-1 f / 2 by Newton with the accumulated gradient and a live sigma
    (what gpb_pref_laplace computes with grad_mode = 1), iterated until max|f_new - f| <= tol."""
    x = np.asarray(x, dtype=float).reshape(len(x), -1)
    D = x.shape[1]
    K = rbf_ard_K(x, np.exp(loghyp[:D]), np.exp(loghyp[D]) ** 2) + eps * np.eye(len(x))
    lik = ProbitPrefOracle(sigma)
    uvi = np.asarray(uvi)
    y = np.asarray(y, dtype=float).reshape(-1, 1)
    iK = np.linalg.inv(K)
    f = np.zeros((len(x), 1))
    for _ in range(max_iter):
        W, g = lik.derivatives(uvi, y, f, accumulate=True)
        f_new = np.linalg.solve(iK + W, W @ f + g)
        err = np.max(np.abs(f_new - f))
        f = f_new
        if err <= tol:
            break
    return f[:, 0]


def laplace_evidence_grad(x, uvi, y, loghyp, f, sigma=1.0, eps=1e-6):
    """(laplace_evidence, d/d[log l_1..log l_D, log sf, log sigma]) at the mode f, with eps held fixed.

    W = sum_k w_k a_k a_k', a_k = y_k s (e_v - e_u), s = 1 / (sqrt(2) sigma), G = K^-1 + W, alpha = K^-1 f,
    A = K^-1 - K^-1 G^-1 K^-1, c_k = a_k' G^-1 a_k, s2 = 1/2 sum_k r2_k c_k a_k, v = G^-1 s2, u = K^-1 v,
    M = A - alpha alpha' - u alpha' - alpha u',   d/dtheta_j = -1/2 tr(M dK/dtheta_j)   (dK/dlog sf = 2 sf2 k_SE),
    h = sum_k (w_k z_k - r_k) a_k,   d/dlog sigma = -sum r z - 1/2 sum (r2 z - 2 w) c + v'h.
    Exact only at a stationary point of sum log Phi - f'K^-1 f / 2 (the accumulated-gradient mode)."""
    x = np.asarray(x, dtype=float).reshape(len(x), -1)
    n, D = x.shape
    uvi = np.asarray(uvi)
    yv = np.asarray(y, dtype=float).reshape(-1)
    f = np.asarray(f, dtype=float).reshape(-1)
    ell = np.exp(loghyp[:D])
    sf2 = np.exp(loghyp[D]) ** 2
    s = 1.0 / (np.sqrt(2.0) * sigma)
    Kse = rbf_ard_K(x, ell, sf2)
    K = Kse + eps * np.eye(n)
    a = np.zeros((len(uvi), n))
    k = np.arange(len(uvi))
    np.add.at(a, (k, uvi[:, 1]), yv * s)
    np.add.at(a, (k, uvi[:, 0]), -yv * s)
    z = a @ f
    r, w, r2 = probit_terms(z)
    W = a.T @ (w[:, None] * a)
    iK = np.linalg.inv(K)
    Gi = np.linalg.inv(iK + W)
    alpha = iK @ f
    A = iK - iK @ Gi @ iK
    c = np.einsum('ki,ij,kj->k', a, Gi, a)
    s2 = 0.5 * a.T @ (r2 * c)
    v = Gi @ s2
    u = iK @ v
    M = A - np.outer(alpha, alpha) - np.outer(u, alpha) - np.outer(alpha, u)
    xs = x / ell
    grad = [-0.5 * np.sum(M * Kse * (xs[:, j, None] - xs[None, :, j]) ** 2) for j in range(D)]
    grad.append(-0.5 * np.sum(M * 2.0 * Kse))
    h = a.T @ (w * z - r)
    grad.append(-np.sum(r * z) - 0.5 * np.sum((r2 * z - 2.0 * w) * c) + v @ h)
    return laplace_evidence(x, uvi, y, loghyp, f, sigma, eps), np.array(grad)
