"""Edge cases of the paths in SURVEY 8(a): tiny / ragged sizes, single test points, duplicated inputs, one pair,
unreferenced items, one-class labels - each against the CPU oracle through the same C-ABI calls."""
import numpy as np
import pytest

from oracle import gpr_oracle, gppref_oracle, gpc_oracle

pytestmark = pytest.mark.gpu


def natural(log_hyp):
    from gptest_b200.sweep import natural_params
    return natural_params(log_hyp)[0]


@pytest.mark.parametrize('n,d', [(1, 1), (2, 3), (127, 2), (128, 2), (129, 2), (255, 9), (257, 17)])
def test_gpr_ragged_sizes(handle, n, d):
    rng = np.random.default_rng(n * 31 + d)
    X = rng.random((n, d))
    y = np.sin(X.sum(1)) + 0.1 * rng.standard_normal(n)
    lh = np.log([0.7] * d + [1.3, 0.2])
    handle.set_train(X, y)
    v = handle.gpr_nlml(natural(lh))
    ref = gpr_oracle.nlml_chol(lh, X, y)
    assert abs(v - ref) <= 1e-8 * max(1.0, abs(ref))
    for m in (1, 65):
        Z = rng.random((m, d))
        fz, cov = handle.gpr_predict(natural(lh), Z)
        rf, rc = gpr_oracle.predict_chol(lh, X, y, Z)
        assert fz.shape == (m,) and np.abs(fz - rf).max() <= 1e-9 * max(1.0, np.abs(rf).max())
        assert np.abs(cov - rc).max() <= 1e-9
    v2, g = handle.gpr_nlml(natural(lh), want_grad=True)
    assert abs(v2 - ref) <= 1e-8 * max(1.0, abs(ref))
    rg = gpr_oracle.nlml_grad(lh, X, y)
    assert np.abs(g - rg).max() <= 1e-7 * max(1.0, np.abs(rg).max())


def test_gpr_duplicated_inputs(handle):
    """Repeated training points: fine with noise, LinAlgError without (np.linalg.cholesky, GPr.py:62)."""
    rng = np.random.default_rng(0)
    X = rng.random((50, 2))
    X = np.vstack([X, X[:20]])
    y = rng.standard_normal(70)
    lh = np.log([0.5, 0.5, 1.0, 0.1])
    handle.set_train(X, y)
    ref = gpr_oracle.nlml_chol(lh, X, y)
    assert abs(handle.gpr_nlml(natural(lh)) - ref) <= 1e-8 * abs(ref)
    with pytest.raises(np.linalg.LinAlgError):
        handle.gpr_nlml(natural(np.log([0.5, 0.5, 1.0, 1e-200])))
    from gptest_b200 import GPr
    gp = GPr.GaussianProcess(lh, 0, 0, "SE", "zero", "zero", X, y)
    with pytest.raises(np.linalg.LinAlgError):
        gp.compute_likelihood(np.log([0.5, 0.5, 1.0, 1e-200]))


def test_gpr_constant_mean_argument(handle):
    rng = np.random.default_rng(2)
    X = rng.random((90, 2))
    y = 5.0 + rng.standard_normal(90)
    lh = np.log([0.5, 0.5, 1.0, 0.3])
    handle.set_train(X, y)
    v = handle.gpr_nlml(natural(lh), mean=5.0)
    ref = gpr_oracle.nlml_chol(lh, X, y - 5.0)
    assert abs(v - ref) <= 1e-9 * abs(ref)


def pref_khyp(loghyp, d):
    return np.concatenate([np.exp(loghyp[:d]), [np.exp(loghyp[d]) ** 2]])


@pytest.mark.parametrize('n,pairs', [
    (2, [(0, 1)]),                                   # one pair, two items
    (9, [(0, 1)]),                                   # items that no pair mentions
    (5, [(0, 1), (0, 1), (1, 0), (2, 3), (0, 1)]),   # repeated and reversed pairs
    (130, [(i, (i * 7 + 1) % 130) for i in range(129)]),   # across a tile boundary
])
def test_pref_small_graphs(handle, n, pairs):
    rng = np.random.default_rng(n)
    x = rng.random((n, 2))
    uvi = np.array(pairs, dtype=np.int64)
    y = np.where(rng.random(len(pairs)) < 0.5, 1.0, -1.0).reshape(-1, 1)
    lh = np.log([0.4, 0.6, 1.1, 0.1])
    handle.set_train(x)
    f, lml, iters, trace, jit = handle.pref_laplace(uvi, y, pref_khyp(lh, 2), sigma=1.0, delta_f=1e-7, max_iter=300)
    of, olml, otrace = gppref_oracle.calc_laplace(x, uvi, y, lh, delta_f=1e-7, max_iter=300, return_trace=True)
    assert iters == len(otrace)
    assert np.abs(f.reshape(-1) - of.reshape(-1)).max() < 1e-6
    assert abs(lml - olml) <= 1e-8 * max(1.0, abs(olml))


@pytest.mark.parametrize('labels', ['all_plus', 'all_minus', 'single_minus'])
def test_gpc_one_sided_labels(handle, labels):
    rng = np.random.default_rng(4)
    n = 140
    x = rng.random((n, 2))
    y = np.ones(n)
    if labels == 'all_minus':
        y = -y
    if labels == 'single_minus':
        y[17] = -1.0
    lh = np.log([0.5, 0.5, 1.0])
    handle.set_train(x)
    kh = np.r_[np.exp(lh[:2]), np.exp(lh[2]) ** 2]
    f, lml, iters, trace, jit = handle.gpc_laplace(y, kh, link=0, delta_f=1e-7)
    of, olml = gpc_oracle.calc_laplace(x, y, lh, delta_f=1e-7)
    assert np.abs(f - of).max() < 1e-6
    assert abs(lml - olml) <= 1e-8 * max(1.0, abs(olml))
    z = rng.random((1, 2))
    mu, var, p = handle.gpc_predict(z)
    omu, ovar, op = gpc_oracle.predict(x, y, lh, z, delta_f=1e-7)
    assert abs(p[0] - op[0]) < 1e-7


def test_laplace_fits_ignore_the_regression_covariance_kind(handle):
    """cov_kind selects the covariance of the regression calls only: a preference and a classification fit after a
    Matern regression call on the handle equal, bit for bit, the same fits after a squared-exponential one."""
    rng = np.random.default_rng(11)
    n = 200
    x = rng.random((n, 2))
    yr = np.sin(3.0 * x.sum(1))
    uvi = np.array([(i, (i * 7 + 3) % n) for i in range(n)], dtype=np.int64)
    yp = np.where(rng.random(n) < 0.5, 1.0, -1.0).reshape(-1, 1)
    yc = np.where(x[:, 0] > 0.5, 1.0, -1.0)
    kh = np.array([0.4, 0.6, 1.1])
    z = rng.random((50, 2))

    def fits(kind):
        handle.set_train(x, yr)
        handle.gpr_nlml(np.r_[kh, 0.01], kind=kind)
        pref = handle.pref_laplace(uvi, yp, kh, sigma=1.0, delta_f=1e-7, max_iter=300)
        pref_pred = handle.pref_predict(z)
        gpc = handle.gpc_laplace(yc, kh, link=0, delta_f=1e-7)
        gpc_pred = handle.gpc_predict(z)
        return [np.asarray(a) for r in (pref, pref_pred, gpc, gpc_pred) for a in r]

    matern = fits(1)
    se = fits(0)
    assert len(matern) == len(se)
    for a, b in zip(matern, se):
        assert np.array_equal(a, b, equal_nan=True)


def test_argument_errors(handle):
    from gptest_b200._lib import GpbError
    X = np.random.default_rng(0).random((10, 2))
    handle.set_train(X)                                  # no targets
    with pytest.raises(GpbError, match='targets'):
        handle.gpr_nlml(np.array([1.0, 1.0, 1.0, 0.1]))
    with pytest.raises(GpbError):
        handle.pref_laplace(np.array([[0, 10]], dtype=np.int64), np.ones((1, 1)), np.array([1.0, 1.0, 1.0]),
                            sigma=1.0, delta_f=1e-6, max_iter=10)      # item index out of range


# ---- other covariance functions behind the string dispatch (SURVEY 8f rank 4; not in the reference) -----------
@pytest.mark.parametrize('name', ['Matern32', 'Matern52'])
@pytest.mark.parametrize('n,d', [(90, 1), (700, 3), (1100, 8)])
def test_matern_paths_match_oracle(handle, name, n, d):
    kind = gpr_oracle.KINDS[name]
    rng = np.random.default_rng(n + d)
    X = rng.random((n, d))
    y = np.sin(X.sum(1)) + 0.1 * rng.standard_normal(n)
    Z = rng.random((77, d))
    lh = np.log([0.7] * d + [1.3, 0.2])
    kh = natural(lh)
    handle.set_train(X, y)
    K = handle.kxx(kh, kind=kind)
    assert np.abs(K - gpr_oracle.kxx_kind(lh, X, name)).max() < 1e-12
    assert np.abs(handle.kxz(kh, Z, kind=kind) - gpr_oracle.kxz_kind(lh, X, Z, name)).max() < 1e-12
    v, g = handle.gpr_nlml(kh, want_grad=True, kind=kind)
    rv, rg = gpr_oracle.nlml_kind(lh, X, y, name, want_grad=True)
    assert abs(v - rv) <= 1e-8 * max(1.0, abs(rv))
    assert np.abs(g - rg).max() <= 1e-7 * max(1.0, np.abs(rg).max())
    assert abs(handle.gpr_nlml(kh, kind=kind) - rv) <= 1e-8 * max(1.0, abs(rv))
    fz, cov = handle.gpr_predict(kh, Z, kind=kind)
    rf, rc = gpr_oracle.predict_kind(lh, X, y, Z, name)
    assert np.abs(fz - rf).max() <= 1e-9 * max(1.0, np.abs(rf).max()) and np.abs(cov - rc).max() <= 1e-9
    vals, info = handle.gpr_nlml_batched(np.array([kh, kh * 1.1]), kind=kind)
    assert abs(vals[0] - rv) <= 1e-8 * max(1.0, abs(rv)) and not info.any()
    # the default stays the reference's kernel
    assert abs(handle.gpr_nlml(kh) - gpr_oracle.nlml_chol(lh, X, y)) <= 1e-8 * max(1.0, abs(rv))


def test_matern_dropin_names_and_growing_set(handle):
    from gptest_b200 import GPr
    rng = np.random.default_rng(8)
    X = rng.random((150, 2))
    y = np.cos(3 * X[:, 0]) + 0.1 * rng.standard_normal(150)
    Z = rng.random((20, 2))
    lh = np.log([0.5, 0.8, 1.0, 0.15])
    gp = GPr.GaussianProcess(lh, 0, 0, "Matern52", "zero", "zero", X, y)
    assert isinstance(gp.covFun, GPr.Matern52)
    v = gp.compute_likelihood(lh)
    assert v.shape == (1, 1) and abs(v[0, 0] - gpr_oracle.nlml_kind(lh, X, y, 'Matern52')) <= 1e-8 * abs(v[0, 0])
    fz, cov = gp.compute_prediction(Z)
    rf, rc = gpr_oracle.predict_kind(lh, X, y, Z, 'Matern52')
    assert np.abs(fz - rf).max() < 1e-9 and np.abs(cov - rc).max() < 1e-9
    assert GPr.GaussianProcess(lh, 0, 0, "nope", "zero", "zero", X, y).covFun == []       # GPr.py:31-32
    handle.grow_begin(natural(lh), 2, capacity=150, kind=1)
    handle.grow_append(X[:100], y[:100])
    v2 = handle.grow_append(X[100:], y[100:])
    assert abs(v2 - gpr_oracle.nlml_kind(lh, X, y, 'Matern32')) <= 1e-8 * abs(v2)
    fz, cov = handle.grow_predict(Z)
    rf, rc = gpr_oracle.predict_kind(lh, X, y, Z, 'Matern32')
    assert np.abs(fz - rf).max() < 1e-9 and np.abs(cov - rc).max() < 1e-9


def test_two_handles_are_independent(handle):
    """Different handles own their work space and streams: interleaved calls must not disturb each other
    (include/gpb200.h: 'different handles are independent')."""
    from gptest_b200 import _lib
    other = _lib.Handle(0)
    try:
        rng = np.random.default_rng(21)
        Xa, Xb = rng.random((500, 3)), rng.random((333, 2))
        ya, yb = np.sin(Xa.sum(1)), np.cos(Xb.sum(1))
        lha, lhb = np.log([0.6] * 3 + [1.0, 0.1]), np.log([0.4] * 2 + [1.2, 0.2])
        handle.set_train(Xa, ya)
        other.set_train(Xb, yb)
        other.grow_begin(natural(lhb), 2, capacity=400)
        other.grow_append(Xb[:200], yb[:200])
        va = handle.gpr_nlml(natural(lha))
        vb = other.gpr_nlml(natural(lhb), kind=1)              # Matern on one handle ...
        va2, ga = handle.gpr_nlml(natural(lha), want_grad=True)  # ... squared exponential on the other
        vg = other.grow_append(Xb[200:], yb[200:])
        assert abs(va - gpr_oracle.nlml_chol(lha, Xa, ya)) <= 1e-8 * abs(va) and abs(va2 - va) <= 1e-12 * abs(va)
        assert abs(vb - gpr_oracle.nlml_kind(lhb, Xb, yb, 'Matern32')) <= 1e-8 * abs(vb)
        assert abs(vg - gpr_oracle.nlml_chol(lhb, Xb, yb)) <= 1e-8 * abs(vg)
        assert np.abs(ga - gpr_oracle.nlml_grad(lha, Xa, ya)).max() <= 1e-7 * max(1.0, np.abs(ga).max())
    finally:
        other.close()


def test_far_apart_points_underflow_to_zero_like_numpy(handle):
    """Scaled distances of several thousand (short length scales, line-search excursions): x = -r^2/2 down to
    -5e7.  numpy's exp returns exactly 0 there (GPr.py:102); the table exp must too - before the clamp its
    integer exponent wrapped and K held huge or negative entries (ADVICE round 1).  The checker is the direct
    difference form: with coordinates of 1e4 length scales the reference's own expanded form (GPr.py:4-13)
    carries eps * |x/l|^2 ~ 1e-8 of cancellation noise, also on its diagonal."""
    rng = np.random.default_rng(7)
    X = 100.0 * rng.random((300, 2))
    y = rng.standard_normal(300)
    eye = np.eye(300, dtype=bool)
    for ell in (0.01, 0.004, 1.0):
        lh = np.log([ell, ell, 1.0, 0.1])
        handle.set_train(X, y)
        K = handle.kxx(natural(lh))
        dif = (X[:, None, :] - X[None, :, :]) / ell
        exact = np.exp(-0.5 * np.sum(dif * dif, axis=2)) + 0.1 ** 2 * np.eye(300)
        assert np.isfinite(K).all() and (K >= 0).all()
        tol = 2e-14 + 8 * 2.3e-16 * (100.0 / ell) ** 2
        assert np.abs(K - exact).max() <= tol
        assert np.abs(K - gpr_oracle.kxx(lh, X)).max() <= 2 * tol          # the reference form, same noise bound
        assert (K[~eye][exact[~eye] == 0.0] == 0.0).all()                  # deep underflow is an exact zero
        assert (exact[~eye] == 0.0).mean() > 0.5
        v = handle.gpr_nlml(natural(lh))
        L = np.linalg.cholesky(exact)
        z = np.linalg.solve(L, y)
        r = 0.5 * z @ z + np.log(np.diag(L)).sum() + 150 * np.log(2 * np.pi)
        assert abs(v - r) <= 1e-8 * abs(r) + 300 * tol
        vg, g = handle.gpr_nlml(natural(lh), want_grad=True)
        assert np.isfinite(g).all() and abs(vg - v) <= 1e-12 * abs(v)
    # Matern kernels go through the same exp with x = -a
    handle.set_train(X, y)
    K = handle.kxx(natural(np.log([1e-4, 1e-4, 1.0, 0.1])), kind=1)
    assert np.isfinite(K).all() and (K[~eye] == 0.0).all() and np.abs(np.diag(K) - 1.01).max() < 1e-15


def test_hyperparameter_vector_of_the_wrong_length_is_refused(handle):
    """A log_hyp that does not fit the input dimension (e.g. the 3-entry demo vector with 2-D X): the reference
    raises a numpy broadcasting ValueError; the binding must not read past the vector."""
    rng = np.random.default_rng(3)
    X = rng.random((40, 2))
    y = rng.standard_normal(40)
    handle.set_train(X, y)
    bad = np.array([0.5, 1.0, 0.01])
    for call in (lambda: handle.gpr_nlml(bad), lambda: handle.gpr_predict(bad, X[:3]), lambda: handle.kxx(bad),
                 lambda: handle.kxz(bad, X[:3]), lambda: handle.gpr_nlml_batched(np.tile(bad, (4, 1))),
                 lambda: handle.gpc_laplace(np.sign(y), np.array([0.5, 1.0])),
                 lambda: handle.pref_laplace(np.array([[0, 1]]), np.array([1.0]), np.array([0.5, 0.5, 1.0, 1.0]))):
        with pytest.raises(ValueError):
            call()
    from gptest_b200 import GPr
    gp = GPr.GaussianProcess(np.log([1.0, 1.0, 0.1]), 0, 0, "SE", "zero", "zero", X, y)
    with pytest.raises(ValueError):
        gp.compute_likelihood(np.log([1.0, 1.0, 0.1]))
    with pytest.raises(ValueError):
        gp.compute_prediction(X[:3])


@pytest.mark.parametrize('opt,val', [('potrf_variant', 2), ('split_tiles', 0), ('lookahead', 0)])
def test_alternative_kernel_paths_agree_with_the_default(handle, opt, val):
    """The kernels kept behind options (the previous register-resident diagonal-tile kernel, 128x128 CTA tiles,
    the plain order) factor the same matrix to rounding."""
    rng = np.random.default_rng(11)
    n = 1536
    M = rng.standard_normal((n, n))
    A = M @ M.T / n + np.eye(n)
    L0 = handle.potrf(A)
    handle.set_option(opt, val)
    try:
        L1 = handle.potrf(A)
    finally:
        handle.set_option(opt, {'potrf_variant': 3, 'split_tiles': 1, 'lookahead': 1}[opt])
    assert np.abs(L0 - np.linalg.cholesky(A)).max() < 1e-12
    assert np.abs(L1 - L0).max() < 1e-12


@pytest.mark.parametrize('bad', [0, 5, 31, 32, 40, 100, 127, 128, 200, 383])
def test_first_failing_pivot_is_reported_like_lapack(handle, bad):
    """np.linalg.cholesky (GPr.py:62) raises on a non-positive pivot; the C ABI reports LAPACK's info = index of the
    first failing leading minor, wherever it falls inside the blocked diagonal-tile kernel (32-blocks, 8-column panels)."""
    n = 384
    rng = np.random.default_rng(bad)
    M = rng.standard_normal((n, n))
    A = M @ M.T / n + np.eye(n)
    # make the leading minor of order bad+1 singular-negative: subtract enough from the diagonal entry
    L = np.linalg.cholesky(A)
    A[bad, bad] -= 1.5 * L[bad, bad] ** 2
    with pytest.raises(np.linalg.LinAlgError) as e:
        handle.potrf(A)
    assert 'leading minor %d)' % (bad + 1) in str(e.value)
    handle.set_option('potrf_variant', 2)
    try:
        with pytest.raises(np.linalg.LinAlgError) as e2:
            handle.potrf(A)
    finally:
        handle.set_option('potrf_variant', 3)
    assert 'leading minor %d)' % (bad + 1) in str(e2.value)
