"""CPU tests of host-side logic that needs no device: the factor-synchronisation rules of the GPy-shaped layer
(with a recording stand-in for the handle), the covariance-name dispatch of the GPr mirror, and a numpy model of the
block append that csrc/grow.cu performs with device kernels."""
import numpy as np
import pytest

from oracle import gpr_oracle


class FakeHandle(object):
    """Records the calls GPRegression._sync_factor makes; keeps the point count like the C side."""

    def __init__(self):
        self.calls = []
        self.n_grow = -1

    def grow_begin(self, khyp, d, capacity, mean=0.0, kind=0):
        self.calls.append(('begin', int(capacity)))
        self.cap = int(capacity)
        self.n_grow = 0

    def grow_append(self, X, y):
        assert self.n_grow + len(y) <= self.cap
        self.calls.append(('append', len(y)))
        self.n_grow += len(y)
        return 0.0

    def grow_size(self):
        return self.n_grow

    def grow_predict(self, Z):
        self.calls.append(('predict', len(Z)))
        return np.zeros(len(Z)), np.ones(len(Z))


@pytest.fixture
def fake(monkeypatch):
    from gptest_b200 import _lib
    h = FakeHandle()
    monkeypatch.setattr(_lib, 'default_handle', lambda device=None: h)
    return h


def test_replay_appends_instead_of_refitting(fake):
    import gptest_b200.gpy_compat as GPy
    rng = np.random.default_rng(0)
    X, Y = rng.random((60, 2)), rng.standard_normal((60, 1))
    gpm = GPy.models.GPRegression(X[:1], Y[:1], GPy.kern.RBF(input_dim=2, variance=10., lengthscale=20.))
    for i in range(40):                                   # GP_parameter_fit.py:60-63
        gpm.set_XY(X[:i + 1], Y[:i + 1])
        m, v = gpm.predict(X[:3])
        assert m.shape == (3, 1) and np.allclose(v, 1.0 + gpm.likelihood.variance)
    kinds = [c[0] for c in fake.calls]
    assert kinds.count('begin') == 1 and kinds.count('append') == 40 and kinds.count('predict') == 40
    assert all(c[1] == 1 for c in fake.calls if c[0] == 'append')
    # same data, same parameters: nothing is appended, the factor is reused
    gpm.predict(X[:3])
    assert [c[0] for c in fake.calls].count('append') == 40
    # a changed parameter, changed data, or shrinking data rebuild the factor
    for change in ('param', 'data', 'shrink'):
        before = [c[0] for c in fake.calls].count('begin')
        if change == 'param':
            gpm.kern.variance = 11.0
        elif change == 'data':
            Y2 = Y.copy(); Y2[3, 0] += 1.0
            gpm.set_XY(X[:40], Y2[:40])
        else:
            gpm.set_XY(X[:10], Y[:10])
        gpm.predict(X[:3])
        assert [c[0] for c in fake.calls].count('begin') == before + 1, change
        assert fake.n_grow == len(gpm.X)


def test_capacity_growth_rebuilds(fake):
    import gptest_b200.gpy_compat as GPy
    rng = np.random.default_rng(1)
    X, Y = rng.random((3000, 2)), rng.standard_normal((3000, 1))
    gpm = GPy.models.GPRegression(X[:100], Y[:100])
    gpm.predict(X[:2])
    cap0 = fake.cap
    assert cap0 >= 1024
    gpm.set_XY(X[:cap0 + 1], Y[:cap0 + 1])               # beyond the capacity chosen at the first fit
    gpm.predict(X[:2])
    assert fake.cap >= cap0 + 1 and fake.n_grow == cap0 + 1
    assert [c[0] for c in fake.calls].count('begin') == 2


def test_covariance_name_dispatch():
    from gptest_b200 import GPr
    x = np.linspace(0, 1, 7)
    lh = np.log([0.5, 1.0, 0.1])
    for name, cls, kind in (("SE", GPr.SquaredExponential, 0), ("Matern32", GPr.Matern32, 1), ("Matern52", GPr.Matern52, 2)):
        gp = GPr.GaussianProcess(lh, 0, 0, name, "zero", "zero", x, x)
        assert type(gp.covFun) is cls and gp.covFun.KIND == kind
        assert np.array_equal(gp.covFun.M, np.exp(lh[:1])) and gp.covFun.sf2 == np.exp(lh[1]) ** 2    # GPr.py:93-97
        assert gp._cov_class() is cls
    gp = GPr.GaussianProcess(lh, 0, 0, "nope", "nope", "nope", x, x)
    assert gp.covFun == [] and gp.meanFun == [] and gp.likeFun == []                                  # GPr.py:31-42
    assert gpr_oracle.KINDS == {"SE": 0, "Matern32": 1, "Matern52": 2}


@pytest.mark.parametrize('n0,m', [(0, 5), (100, 28), (128, 1), (130, 3), (200, 300)])
def test_block_append_model(n0, m):
    """The algebra of csrc/grow.cu in numpy: with r0 = the start of the 128-tile holding the first new point,
    X = K21 L11^-T, S = K22 - X X^T, L22 = chol(S), z2 = L22^-1 (y2 - X z1) extends the factor of the prefix."""
    rng = np.random.default_rng(n0 + m)
    n1 = n0 + m
    x = rng.random((n1, 2))
    y = rng.standard_normal(n1)
    lh = np.log([0.4, 0.6, 1.0, 0.2])
    K = gpr_oracle.kxx(lh, x)
    L_full = np.linalg.cholesky(K)
    z_full = np.linalg.solve(L_full, y)
    r0 = (n0 // 128) * 128
    L = np.zeros((n1, n1))
    z = np.zeros(n1)
    if n0 > 0:
        L[:n0, :n0] = np.linalg.cholesky(K[:n0, :n0])
        z[:n0] = np.linalg.solve(L[:n0, :n0], y[:n0])
    # everything from row r0 on is rebuilt (rows r0..n0 keep their part left of r0 - recomputing it is the same)
    L11 = L[:r0, :r0]
    Xb = np.linalg.solve(L11, K[r0:, :r0].T).T if r0 else np.zeros((n1 - r0, 0))
    S = K[r0:, r0:] - Xb @ Xb.T
    L[r0:, :r0] = Xb
    L[r0:, r0:] = np.linalg.cholesky(S)
    z[r0:] = np.linalg.solve(L[r0:, r0:], y[r0:] - Xb @ z[:r0])
    assert np.abs(L - L_full).max() < 1e-12 and np.abs(z - z_full).max() < 1e-11
    nlml = 0.5 * z @ z + np.sum(np.log(np.diag(L))) + n1 * np.log(2 * np.pi) / 2
    assert abs(nlml - gpr_oracle.nlml_chol(lh, x, y)) < 1e-9 * max(1.0, abs(nlml))


def test_gppref_module_level_names_of_the_reference():
    """GPpref.py defines std_norm_pdf, squared_distance, SquaredExponential, PrefProbit and
    PreferenceGaussianProcess at module level; `from GPpref import squared_distance` must keep working."""
    import numpy as np
    from gptest_b200 import GPpref
    for name in ('std_norm_pdf', 'squared_distance', 'SquaredExponential', 'PrefProbit', 'PreferenceGaussianProcess'):
        assert hasattr(GPpref, name), name
    se = GPpref.SquaredExponential(np.log([0.5, 0.5, 1.0]), np.zeros((4, 2)))       # GPpref.py:26-31
    assert se.length.shape == (2,) and abs(se.logvar - 1.0) < 1e-15
    import pytest
    with pytest.raises(AttributeError):                                             # GPpref.py:34 reads self.M
        se.compute_Kxx_matrix()


def test_newton_loop_bodies_have_no_host_round_trip():
    """SURVEY 8(b): 'internal Laplace iterations never sync with host'.  Structural check of csrc/laplace.cu: both
    Newton iterations are lambdas handed to run_device_loop (body of a CUDA-graph WHILE node), factor and end with a
    finish kernel, and contain no synchronisation, no device-to-host copy and no host read."""
    import os
    import re
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gptest_b200', 'csrc', 'laplace.cu')).read()
    # the lambda argument of every run_device_loop call, whatever its parameter list, up to its closing line
    bodies = re.findall(r'run_device_loop\(h, [^\[]*\[&\]\([^)]*cudaGraphConditionalHandle cond\) \{(.*?)\n  \}\);', src, re.S)
    assert len(bodies) == 2
    for b in bodies:
        assert re.search(r'chol_sweep\(h, \w+, true\)', b) and 'finish_kernel' in b
        for banned in ('cudaStreamSynchronize', 'cudaDeviceSynchronize', 'cudaMemcpy', 'read_info', 'pinned(', 'cudaEventSynchronize'):
            assert banned not in b, banned
    assert 'cudaGraphSetConditional' in src and 'cudaGraphCondTypeWhile' in src
