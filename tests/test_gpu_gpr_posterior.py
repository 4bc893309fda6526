"""GPU tests of the joint posterior covariance and the posterior samples of GP regression (gpb_gpr_predict_full,
gpb_gpr_sample) against the Cholesky form of the CPU oracle and the numpy restatement of the generator."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import bench_configs as cfg
from oracle import gpr_oracle
from tests import _posterior_oracle as po

pytestmark = pytest.mark.gpu
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'gpr_kat.json')))
KIND_ID = {'SE': 0, 'Matern32': 1, 'Matern52': 2}


def khyp_of(log_hyp):
    ell, sf2, sn2 = gpr_oracle.split_hyp(log_hyp)
    return np.concatenate([ell, [sf2, sn2]])


def problem(n, d, m, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    y = np.sin(X @ rng.standard_normal(d)) + 0.1 * rng.standard_normal(n)
    Z = rng.random((m, d))
    lh = np.log([0.6] * d + [1.3, 0.2])
    return X, y, Z, lh


def check_full(handle, X, y, Z, lh, kind='SE', noisy=False):
    handle.set_train(X, y)
    kh = khyp_of(lh)
    fz, cov = handle.gpr_predict_full(kh, Z, kind=KIND_ID[kind], noisy=noisy)
    mu, var = handle.gpr_predict(kh, Z, kind=KIND_ID[kind])
    sf2 = kh[-2]
    assert np.array_equal(fz, mu)                                   # the same code, the same bits
    np.testing.assert_array_equal(cov, cov.T)
    extra = kh[-1] if noisy else 0.0
    assert np.max(np.abs(np.diag(cov) - extra - var)) <= 1e-11 * sf2
    _, ref = po.predict_full_chol(lh, X, y, Z, kind, noisy=noisy)
    err = np.max(np.abs(cov - ref))
    assert err <= 1e-9 * sf2, err
    return fz, cov


CASES = [  # n, d, m, kind, noisy
    (300, 1, 1, 'SE', False),
    (300, 2, 77, 'SE', True),
    (300, 8, 129, 'Matern32', False),
    (1000, 2, 300, 'Matern52', True),
    (1000, 8, 1024, 'SE', False),
    (1000, 1, 129, 'Matern32', True),
    (2048, 2, 1024, 'Matern52', False),
    (2048, 8, 300, 'SE', True),
    (2048, 8, 77, 'Matern52', False),
]


@pytest.mark.parametrize("n,d,m,kind,noisy", CASES)
def test_predict_full_matches_oracle(handle, n, d, m, kind, noisy):
    X, y, Z, lh = problem(n, d, m, seed=n + 7 * d + m)
    check_full(handle, X, y, Z, lh, kind, noisy)


@pytest.mark.parametrize("noisy", [False, True])
def test_predict_full_kat1(handle, noisy):
    k = GOLD['kat1']
    check_full(handle, np.array(k['x']).reshape(-1, 1), np.array(k['y']), np.array(k['z']).reshape(-1, 1),
               np.array(k['log_hyp']), noisy=noisy)


def test_predict_full_c2(handle):
    X, y, Z, lh = cfg.make_c2(m=2048)
    check_full(handle, X, y, Z, lh)


def test_predict_full_to_device_memory(handle):
    import torch
    X, y, Z, lh = problem(300, 2, 200, seed=1)
    handle.set_train(X, y)
    kh = khyp_of(lh)
    fz_h, cov_h = handle.gpr_predict_full(kh, Z)
    out = torch.full((200, 200), float('nan'), dtype=torch.float64, device='cuda')
    fz = np.empty(200)
    info = C.c_int32()
    torch.cuda.synchronize()
    handle.check(handle.lib.gpb_gpr_predict_full(handle.h, kh.ctypes.data_as(C.POINTER(C.c_double)), 0.0,
                                                 np.ascontiguousarray(Z).ctypes.data_as(C.POINTER(C.c_double)), 200,
                                                 fz.ctypes.data_as(C.POINTER(C.c_double)), C.c_void_p(out.data_ptr()),
                                                 1, 0, C.byref(info)))
    torch.cuda.synchronize()
    assert info.value == 0
    assert np.array_equal(out.cpu().numpy(), cov_h) and np.array_equal(fz, fz_h)


@pytest.mark.parametrize("m", [256, 300])
def test_samples_recover_factor_and_product(handle, m):
    X, y, Z, lh = problem(500, 2, m, seed=m)
    Z = 3.0 * Z                       # some points outside the data: a well-conditioned posterior covariance
    handle.set_train(X, y)
    kh = khyp_of(lh)
    sf2 = kh[-2]
    fz, cov = handle.gpr_predict_full(kh, Z, noisy=True)
    seed = 0x1234_5678_9abc_def0
    s, jit = handle.gpr_sample(kh, Z, m, seed=seed, noisy=True)
    assert s.shape == (m, m)
    E = po.philox_normals(seed, m, m)
    Lt = np.linalg.solve(E, s - fz)
    assert np.max(np.abs(np.tril(Lt, -1))) <= 1e-9 * np.sqrt(sf2)
    err = np.max(np.abs(Lt.T @ Lt - (cov + jit * np.eye(m))))
    assert err <= 1e-9 * sf2, err


def test_generator_on_the_device(handle):
    rng = np.random.default_rng(5)
    X = rng.random((50, 1))
    handle.set_train(X, rng.standard_normal(50))
    ell = 0.5
    kh = np.array([ell, 4.0, 0.01])
    far = lambda k: (1e4 + 1e3 * ell * np.arange(k)).reshape(-1, 1)   # Sigma* = sf2 I exactly, fz = 0
    seed = 987654321987
    s, jit = handle.gpr_sample(kh, far(333), 5, seed=seed)
    assert jit == 0.0
    np.testing.assert_allclose(s, 2.0 * po.philox_normals(seed, 5, 333), rtol=1e-14, atol=0)
    s2, _ = handle.gpr_sample(kh, far(1000), 5, seed=seed)
    assert np.array_equal(s2[:, :333], s)
    s3, _ = handle.gpr_sample(kh, far(333), 200, seed=seed)
    assert np.array_equal(s3[:5], s)


def test_sample_statistics(handle):
    X, y, Z, lh = problem(400, 2, 64, seed=11)
    Z = 2.0 * Z
    handle.set_train(X, y)
    kh = khyp_of(lh)
    fz, cov = handle.gpr_predict_full(kh, Z)
    S = 100000
    s, jit = handle.gpr_sample(kh, Z, S, seed=77)
    C_ = cov + jit * np.eye(64)
    dm = s.mean(axis=0) - fz
    assert np.all(np.abs(dm) <= 6 * np.sqrt(np.diag(C_) / S))
    Sc = np.cov(s, rowvar=False)
    dg = np.diag(C_)
    se = np.sqrt((np.outer(dg, dg) + C_ ** 2) / S)
    assert np.all(np.abs(Sc - C_) <= 6 * se)


def test_sample_determinism(handle):
    X, y, Z, lh = problem(300, 2, 100, seed=3)
    handle.set_train(X, y)
    kh = khyp_of(lh)
    a, _ = handle.gpr_sample(kh, Z, 16, seed=42)
    b, _ = handle.gpr_sample(kh, Z, 16, seed=42)
    c, _ = handle.gpr_sample(kh, Z, 16, seed=43)
    assert np.array_equal(a, b)
    assert not np.any(a == c)


def test_jitter_policy(handle):
    X, y, Z, lh = problem(300, 2, 40, seed=9)
    Zd = np.vstack([Z, Z, Z])                 # duplicated points: Sigma* is singular
    handle.set_train(X, y)
    kh = khyp_of(lh)
    sf2 = kh[-2]
    _, jit = handle.gpr_sample(kh, Zd, 8, seed=1)
    allowed = sf2 * 10.0 ** np.arange(-12, 1)
    assert jit > 0 and np.min(np.abs(allowed - jit) / allowed) <= 1e-15
    _, jit2 = handle.gpr_sample(kh, Zd, 8, seed=1, noisy=True)
    assert jit2 == 0.0


def test_errors_and_state(handle):
    from gptest_b200._lib import GpbError
    rng = np.random.default_rng(2)
    X = rng.random((70, 2))
    X[50:] = X[:20]
    y = rng.standard_normal(70)
    handle.set_train(X, y)
    bad = np.array([0.5, 0.5, 1.0, 1e-200])               # duplicated training points without noise
    Z = rng.random((30, 2))
    with pytest.raises(np.linalg.LinAlgError):
        handle.gpr_predict_full(bad, Z)
    with pytest.raises(np.linalg.LinAlgError):
        handle.gpr_sample(bad, Z, 4)
    kh = np.array([0.5, 0.5, 1.0, 0.01])
    dp = C.POINTER(C.c_double)
    out = np.empty((4, 30))
    fz = np.empty(30)
    jit = C.c_double()
    info = C.c_int32()
    lib, h = handle.lib, handle.h
    Zc = np.ascontiguousarray(Z)
    args = (kh.ctypes.data_as(dp), 0.0, Zc.ctypes.data_as(dp))
    assert lib.gpb_gpr_sample(h, *args, 30, 0, 1, 0, out.ctypes.data_as(dp), C.byref(jit), C.byref(info)) < 0
    assert lib.gpb_gpr_sample(h, *args, 0, 4, 1, 0, out.ctypes.data_as(dp), C.byref(jit), C.byref(info)) < 0
    assert lib.gpb_gpr_sample(h, *args, 30, 4, 1, 0, None, C.byref(jit), C.byref(info)) < 0
    assert lib.gpb_gpr_sample(None, *args, 30, 4, 1, 0, out.ctypes.data_as(dp), C.byref(jit), C.byref(info)) < 0
    assert lib.gpb_gpr_predict_full(h, *args, -1, fz.ctypes.data_as(dp), out.ctypes.data_as(C.c_void_p), 0, 0,
                                    C.byref(info)) < 0
    assert lib.gpb_gpr_predict_full(h, kh.ctypes.data_as(dp), 0.0, None, 30, fz.ctypes.data_as(dp),
                                    out.ctypes.data_as(C.c_void_p), 0, 0, C.byref(info)) < 0
    assert lib.gpb_gpr_predict_full(h, *args, 30, None, out.ctypes.data_as(C.c_void_p), 0, 0, C.byref(info)) < 0
    # the calls use the work space: a Laplace state is invalidated, the growing-set state is not
    handle.grow_begin(kh, 2, 256)
    handle.grow_append(X[:40], y[:40])
    g0 = handle.grow_predict(Z)
    yc = np.where(y > 0, 1.0, -1.0)
    handle.set_train(X[:40], yc[:40])
    handle.gpc_laplace(yc[:40], np.array([0.4, 0.4, 1.0]))
    handle.gpc_predict(Z)
    handle.gpr_sample(kh, Z, 4)
    with pytest.raises(GpbError):
        handle.gpc_predict(Z)
    handle.gpr_predict_full(kh, Z)
    g1 = handle.grow_predict(Z)
    assert np.array_equal(g0[0], g1[0]) and np.array_equal(g0[1], g1[1])


def test_gpr_module_full_cov_and_samples(handle):
    from gptest_b200 import GPr
    X, y, Z, lh = problem(200, 2, 50, seed=21)
    gp = GPr.GaussianProcess(lh, 0, 0, "SE", "zero", "zero", X, y)
    fz0, var0 = gp.compute_prediction(Z)
    fz, cov = gp.compute_prediction(Z, full_cov=True)
    assert cov.shape == (50, 50) and np.array_equal(fz, fz0)
    assert np.max(np.abs(np.diag(cov) - var0)) <= 1e-11 * np.exp(2 * lh[-2])
    s = gp.compute_posterior_samples(Z, 7, seed=3)
    assert s.shape == (7, 50)
    assert np.array_equal(s, gp.compute_posterior_samples(Z, 7, seed=3))


def test_gpy_compat_full_cov_and_samples(handle):
    from gptest_b200 import gpy_compat as GPy
    rng = np.random.RandomState(0)
    X = rng.uniform(0., 100., (150, 2))
    Y = np.sin(X[:, :1] / 15.0) + 0.25 * rng.randn(150, 1)
    gpm = GPy.models.GPRegression(X, Y, GPy.kern.RBF(input_dim=2, variance=10., lengthscale=20.))
    gpm.likelihood.variance = 0.0625
    Xn = rng.uniform(0., 100., (60, 2))
    mu, var = gpm.predict(Xn)
    mu_f, cov_f = gpm.predict(Xn, full_cov=True)
    assert mu_f.shape == (60, 1) and cov_f.shape == (60, 60)
    np.testing.assert_allclose(np.diag(cov_f), var[:, 0], rtol=1e-9)
    np.testing.assert_allclose(mu_f, mu, rtol=1e-9, atol=1e-12)
    _, cov_nl = gpm.predict_noiseless(Xn, full_cov=True)
    np.testing.assert_allclose(cov_f - cov_nl, 0.0625 * np.eye(60), rtol=0, atol=1e-12)
    np.random.seed(5)
    a = gpm.posterior_samples_f(Xn, size=12)
    np.random.seed(5)
    b = gpm.posterior_samples_f(Xn, size=12)
    assert a.shape == (60, 1, 12) and np.array_equal(a, b)
    assert gpm.posterior_samples(Xn, size=3).shape == (60, 1, 3)
