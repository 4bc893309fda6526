"""Extended-precision reference for the factorisation, the solves and the gradient (test helper, not collected).

Everything here treats the given float64 matrix as EXACT input and computes in ``np.longdouble`` (80-bit extended on
x86-64: eps 1.1e-19, 2048 times finer than float64).  At cond(K) <= 1e12 that leaves the reference about three orders
of magnitude more accurate than any float64 solver of the same matrix; tests/test_xprec_reference.py checks this
against 50-digit mpmath.  Comparing a device result with numpy's own K is hopeless at that conditioning: one ulp of
difference per entry of K, moved through cond(K), is already larger than the answer's tolerance.  So the GPU tests
hand the device's OWN matrix (``Handle.kxx`` / ``Handle.kxz``) to this module.

Three solvers of the same quantities live here:
  * ``Exact``       long-double Cholesky, substitutions, K^-1: the truth;
  * ``Lapack``      float64 LAPACK (scipy cho_factor / cho_solve / solve_triangular): the accuracy a float64 solver
                    of the same matrix reaches, i.e. the envelope the device is held to;
  * ``emulate_chol`` a float64 CPU model of the device's ORDER of operations (128-tiles, 32-blocks factored and
                    inverted, TRSM as a product with the inverted diagonal block, forward solve as z = W r): what
                    the design costs, separately from what the kernels do.

Hyper-parameters are the natural ones of the C ABI, khyp = [l_1..l_D, sf2, sn2]; gradients are with respect to the
log hyper-parameters [log l_1..l_D, log sf, log sn] (include/gpb200.h).
"""
import numpy as np
import scipy.linalg as sla
from threadpoolctl import threadpool_limits

LD = np.longdouble
U = 2.0 ** -53                                      # unit round-off of float64
LOG_2PI = np.log(LD(2)) + np.log(LD('3.14159265358979323846264338327950288'))


def ld_eps():
    return float(np.finfo(LD).eps)


# ---------------------------------------------------------------------------------------------------------------------
# long-double kernels
# ---------------------------------------------------------------------------------------------------------------------
def chol_ld(A):
    """Right-looking Cholesky in long double, one column per step (rank-1 update of the trailing matrix)."""
    A = np.array(A, dtype=LD)
    n = A.shape[0]
    for k in range(n):
        p = A[k, k]
        if not p > 0:
            raise np.linalg.LinAlgError('long-double Cholesky: pivot %d is %r' % (k + 1, p))
        l = np.sqrt(p)
        A[k, k] = l
        c = A[k + 1:, k]
        c /= l
        A[k + 1:, k + 1:] -= np.multiply.outer(c, c)
    return np.tril(A)


def fsub_ld(L, B):
    """Solve L X = B (L lower triangular, long double), row by row."""
    B = np.array(B, dtype=LD)
    vec = B.ndim == 1
    X = B.reshape(len(B), -1).copy()
    for i in range(len(X)):
        if i:
            X[i] -= L[i, :i] @ X[:i]
        X[i] /= L[i, i]
    return X[:, 0] if vec else X


def bsub_ld(L, B):
    """Solve L^T X = B (L lower triangular, long double), row by row from the bottom."""
    B = np.array(B, dtype=LD)
    vec = B.ndim == 1
    X = B.reshape(len(B), -1).copy()
    n = len(X)
    for i in range(n - 1, -1, -1):
        if i < n - 1:
            X[i] -= L[i + 1:, i] @ X[i + 1:]
        X[i] /= L[i, i]
    return X[:, 0] if vec else X


def tril_inv_ld(L):
    """L^-1 of a lower-triangular long-double L (forward substitution on the identity, lower part only)."""
    n = len(L)
    X = np.zeros((n, n), dtype=LD)
    for i in range(n):
        if i:
            X[i, :i] = -(L[i, :i] @ X[:i, :i])
        X[i, i] = 1
        X[i, :i + 1] /= L[i, i]
    return X


def llt_residual(L, A, blk=128):
    """max |L L^T - A| / max |A| over the lower triangle, in long double (L, A: float64 or long double).
    Block rows of the product only run over k <= the block's last row: n^3/3 multiply-adds."""
    L = np.asarray(L, dtype=LD)
    A = np.asarray(A, dtype=LD)
    n = len(A)
    worst = LD(0)
    for r0 in range(0, n, blk):
        r1 = min(n, r0 + blk)
        R = L[r0:r1, :r1] @ L[:r1, :r1].T - A[r0:r1, :r1]
        R = np.tril(R, r0)                         # columns 0..row of each row
        worst = max(worst, np.abs(R).max())
    return float(worst / np.abs(A).max())


def se_dK(X, khyp, K):
    """dK/dtheta for theta = [log l_1..l_D, log sf, log sn] of the squared exponential, from the GIVEN matrix K:
    K_se = K - sn2 I, dK/dlog l_k = K_se o (x_ik - x_jk)^2 / l_k^2, dK/dlog sf = 2 K_se, dK/dlog sn = 2 sn2 I.
    Returned as (list of D dense matrices, K_se, sn2), all in the dtype of K."""
    dt = K.dtype
    X = np.asarray(X, dtype=np.float64).reshape(len(X), -1)
    khyp = np.asarray(khyp, dtype=np.float64)
    d = X.shape[1]
    sn2 = dt.type(khyp[d + 1])
    Kse = K.copy()
    Kse[np.diag_indices(len(K))] -= sn2
    dl = []
    for k in range(d):
        xs = X[:, k].astype(dt) / dt.type(khyp[k])
        dl.append(Kse * (xs[:, None] - xs[None, :]) ** 2)
    return dl, Kse, sn2


def _grad(Kinv, alpha, dl, Kse, sn2):
    Q = Kinv - np.multiply.outer(alpha, alpha)
    g = [0.5 * np.sum(Q * D) for D in dl]
    g.append(np.sum(Q * Kse))                       # 0.5 tr(Q 2 K_se)
    g.append(np.trace(Q) * sn2)                     # 0.5 tr(Q 2 sn2 I)
    return np.array(g)


# ---------------------------------------------------------------------------------------------------------------------
# the two solvers of one matrix
# ---------------------------------------------------------------------------------------------------------------------
class Exact:
    """Long-double Cholesky of the float64 matrix K (exact input) and the quantities built on it."""
    dtype = LD

    def __init__(self, K):
        self.K = np.asarray(K, dtype=np.float64)
        self.n = len(K)
        self.L = chol_ld(self.K)
        self._Kinv = None

    def logdet_half(self):
        return np.sum(np.log(np.diagonal(self.L)))

    def z(self, r):
        return fsub_ld(self.L, r)

    def alpha(self, r):
        return bsub_ld(self.L, self.z(r))

    def nlml(self, y, mean=0.0):
        z = self.z(np.asarray(y, dtype=LD) - LD(mean))
        return 0.5 * (z @ z) + self.logdet_half() + self.n * LOG_2PI / 2

    def predict(self, y, Kxz, sf2, mean=0.0):
        """Posterior mean (without the constant mean added back, like GPr.py:52) and latent variance sf2 - diag(Kzx K^-1 Kxz)."""
        Kxz = np.asarray(Kxz, dtype=LD)
        alpha = self.alpha(np.asarray(y, dtype=LD) - LD(mean))
        V = fsub_ld(self.L, Kxz)
        return Kxz.T @ alpha, LD(sf2) - np.sum(V * V, axis=0)

    def kinv(self):
        if self._Kinv is None:
            W = tril_inv_ld(self.L)
            self._Kinv = W.T @ W
        return self._Kinv

    def se_grad(self, X, y, khyp, mean=0.0):
        K = self.K.astype(LD)
        dl, Kse, sn2 = se_dK(X, khyp, K)
        return _grad(self.kinv(), self.alpha(np.asarray(y, dtype=LD) - LD(mean)), dl, Kse, sn2)

    def posterior_cov(self, Kxz, Kzz):
        """Sigma* = Kzz - V^T V, V = L^-1 Kxz: the joint posterior covariance of the test points (Kzz given, with
        sn2 on its diagonal for the noisy predictive)."""
        V = fsub_ld(self.L, Kxz)
        return np.asarray(Kzz, dtype=LD) - V.T @ V


def one_blas_thread():
    """LAPACK's rounding depends on how the BLAS splits its sums, i.e. on the thread count: pin it so that the
    envelope is the same on every host."""
    return threadpool_limits(1, user_api='blas')


class Lapack:
    """The same quantities from float64 LAPACK on the same matrix: the envelope the device is held to.
    Call its methods under ``one_blas_thread()`` (``lapack_samples`` does)."""
    dtype = np.float64

    def __init__(self, K):
        self.K = np.asarray(K, dtype=np.float64)
        self.n = len(K)
        with one_blas_thread():
            self.L = np.tril(sla.cho_factor(self.K, lower=True)[0])

    def logdet_half(self):
        return np.sum(np.log(np.diagonal(self.L)))

    def z(self, r):
        return sla.solve_triangular(self.L, r, lower=True)

    def alpha(self, r):
        return sla.cho_solve((self.L, True), r)

    def nlml(self, y, mean=0.0):
        z = self.z(np.asarray(y, dtype=np.float64) - mean)
        return 0.5 * (z @ z) + self.logdet_half() + self.n * np.log(2 * np.pi) / 2

    def predict(self, y, Kxz, sf2, mean=0.0):
        alpha = self.alpha(np.asarray(y, dtype=np.float64) - mean)
        V = sla.solve_triangular(self.L, Kxz, lower=True)
        return Kxz.T @ alpha, sf2 - np.sum(V * V, axis=0)

    def kinv(self):
        return sla.cho_solve((self.L, True), np.eye(self.n))

    def se_grad(self, X, y, khyp, mean=0.0):
        dl, Kse, sn2 = se_dK(X, khyp, self.K.copy())
        return _grad(self.kinv(), self.alpha(np.asarray(y, dtype=np.float64) - mean), dl, Kse, sn2)

    def posterior_cov(self, Kxz, Kzz):
        V = sla.solve_triangular(self.L, Kxz, lower=True)
        return Kzz - V.T @ V


# ---------------------------------------------------------------------------------------------------------------------
# the acceptance criterion
# ---------------------------------------------------------------------------------------------------------------------
N_PERM = 5


def permutations(n, k=N_PERM, seed=0):
    """The identity and k - 1 seeded random orderings of n points."""
    rng = np.random.default_rng(seed)
    return [np.arange(n)] + [rng.permutation(n) for _ in range(k - 1)]


def lapack_samples(K, f, k=N_PERM):
    """f(Lapack(P K P^T), p) for the identity and k - 1 random symmetric permutations p.  Relabelling the training
    points changes nothing in exact arithmetic (f gets p to permute y, X, Kxz alike) but everything about LAPACK's
    rounding: one LAPACK run on one matrix can be lucky by 10-40x on a value that is a sum of cancelling terms, and
    the envelope should not be fitted to that luck."""
    out = []
    with one_blas_thread():
        for p in permutations(len(K), k):
            out.append(f(Lapack(K[np.ix_(p, p)]), p))
    return out


def forward_check(got, lapack, truth, n, scale, factor=10.0):
    """C1: max|got - truth| <= factor * err_lapack + 16 n u scale, err_lapack = max|lapack - truth|; ``lapack`` may
    be a list of samples (``lapack_samples``), err_lapack is then their median.
    Returns (ok, ratio, err_got, err_lapack) with ratio = err_got / err_lapack (inf if LAPACK is exact)."""
    t = np.asarray(truth, dtype=LD)
    eg = float(np.max(np.abs(np.asarray(got, dtype=LD) - t)))
    samples = lapack if isinstance(lapack, list) else [lapack]
    el = float(np.median([float(np.max(np.abs(np.asarray(v, dtype=LD) - t))) for v in samples]))
    ok = eg <= factor * el + 16 * n * U * float(scale)
    ratio = eg / el if el > 0 else (0.0 if eg == 0 else float('inf'))
    return ok, ratio, eg, el


def backward_bound(n):
    """C2: the factor's backward error max|L L^T - A| / max|A| may be at most 4 n u."""
    return 4 * n * U


# ---------------------------------------------------------------------------------------------------------------------
# the sampler's factor, seen through its draws
# ---------------------------------------------------------------------------------------------------------------------
def recover_factor(E, D):
    """The least-squares L of E L^T = D (E: S x m normals with S >= m, D: S x m draws) in long double, through the
    normal equations (E^T E) L^T = E^T D factored by chol_ld.  With S = 4 m, E is well conditioned (cond(E^T E) ~ 10)
    and the recovered factor's backward error is within a few per cent of the true factor's (test_xprec_reference)."""
    E = np.asarray(E, dtype=LD)
    C = chol_ld(E.T @ E)
    return bsub_ld(C, fsub_ld(C, E.T @ np.asarray(D, dtype=LD))).T


def ld_factors(A):
    """True when the long-double Cholesky of A runs to the end (every pivot positive)."""
    try:
        chol_ld(A)
    except np.linalg.LinAlgError:
        return False
    return True


# ---------------------------------------------------------------------------------------------------------------------
# CPU model of the device's order of operations (float64)
# ---------------------------------------------------------------------------------------------------------------------
def _block_factor_inverse(A, blk):
    """Factor and invert one diagonal tile the way tile_potrf3.cu does: 32-blocks factored (Cholesky) and inverted
    (substitution on the identity, the augmented sweep), X = A_ij W_jj^T for the blocks below, A_il -= X_i X_l^T, and
    the off-diagonal blocks of the inverse W_ij = -W_ii (sum_{m=j}^{i-1} L_im W_mj)."""
    A = np.array(A, dtype=np.float64)
    t = len(A)
    nb = t // blk
    W = np.zeros_like(A)
    for j in range(nb):
        sj = slice(j * blk, (j + 1) * blk)
        Ljj = np.linalg.cholesky(A[sj, sj])
        A[sj, sj] = Ljj
        W[sj, sj] = sla.solve_triangular(Ljj, np.eye(blk), lower=True)
        below = slice((j + 1) * blk, t)
        A[below, sj] = A[below, sj] @ W[sj, sj].T
        A[below, below] -= A[below, sj] @ A[below, sj].T
    for i in range(nb):
        si = slice(i * blk, (i + 1) * blk)
        for j in range(i):
            sj = slice(j * blk, (j + 1) * blk)
            S = sum(A[si, m * blk:(m + 1) * blk] @ W[m * blk:(m + 1) * blk, sj] for m in range(j, i))
            W[si, sj] = -W[si, si] @ S
    return np.tril(A), W


def emulate_chol(K, r, tile=128, blk=32, unstable_w=False):
    """Blocked Cholesky of K in the device's order, with the forward solve z = L^-1 r riding on it (z_k = W_kk r_k,
    r_below -= X z_k).  Returns (L, z) for the leading n rows (K is padded with the identity to whole tiles).
    unstable_w: form each tile's inverse as W = L^T (L L^T)^-1 instead, which squares the tile's condition number."""
    n = len(K)
    npad = -(-n // tile) * tile
    A = np.eye(npad)
    A[:n, :n] = K
    rr = np.zeros(npad)
    rr[:n] = r
    z = np.zeros(npad)
    for k in range(npad // tile):
        sk = slice(k * tile, (k + 1) * tile)
        below = slice((k + 1) * tile, npad)
        Lkk, Wkk = _block_factor_inverse(A[sk, sk], blk)
        if unstable_w:
            Wkk = Lkk.T @ np.linalg.inv(Lkk @ Lkk.T)
        A[sk, sk] = Lkk
        z[sk] = Wkk @ rr[sk]
        X = A[below, sk] @ Wkk.T
        A[below, sk] = X
        A[below, below] -= X @ X.T
        rr[below] -= X @ z[sk]
    return np.tril(A)[:n, :n], z[:n]


def gp_inputs(fam, n, sn, seed=None):
    """(X, y, Z, khyp, kind) of the GP families of the conditioning tests; khyp natural [l.., sf2, sn2].
    F1 squared exponential on dense 1-D inputs (l = 0.3), F2 the same with D = 8 (l = 0.5), F3 Matern 3/2 (kind 1),
    F5 Matern 5/2 (kind 2); F3 and F5 have F1's inputs."""
    rng = np.random.default_rng(n if seed is None else seed)
    d = 8 if fam == 'F2' else 1
    X = rng.random((n, d))
    y = np.sin(6 * X.sum(1) / d) + 0.1 * rng.standard_normal(n)
    Z = rng.random((50, d))
    ell = 0.5 if fam == 'F2' else 0.3
    return X, y, Z, np.r_[[ell] * d, 1.0, sn * sn], {'F3': 1, 'F5': 2}.get(fam, 0)


def posterior_points(X, m, seed=0):
    """m test points of the posterior checks, three kinds in turn: uniform in the data box [0, 1)^d; exact copies of
    distinct training rows, where Sigma* = O(sn2) and the cancellation in Kzz - V^T V is largest; and points in
    [2, 3)^d outside the box, where Sigma* is close to Kzz."""
    rng = np.random.default_rng(seed)
    n, d = X.shape
    kind = np.arange(m) % 3
    Z = rng.random((m, d))
    copies = np.flatnonzero(kind == 1)
    Z[copies] = X[rng.choice(n, len(copies), replace=len(copies) > n)]
    Z[kind == 2] += 2.0
    return Z


def emulate_nlml(K, y, **kw):
    L, z = emulate_chol(K, np.asarray(y, dtype=np.float64), **kw)
    return 0.5 * (z @ z) + np.sum(np.log(np.diagonal(L))) + len(K) * np.log(2 * np.pi) / 2, L
