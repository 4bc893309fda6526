"""GPU parity tests of the Laplace paths (GPpref.py:46-161, GPc.py intent) vs the CPU oracles.

Tolerance (north_star): 1e-6 on the Laplace mode after the same iteration count; 1e-8 relative on
the log marginal likelihood."""
import os

import numpy as np
import pytest

from oracle import gppref_oracle, gpc_oracle

pytestmark = pytest.mark.gpu
PREF = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'gppref_kat.npz'))


def pref_khyp(loghyp, d):
    return np.concatenate([np.exp(loghyp[:d]), [np.exp(loghyp[d]) ** 2]])


def make_pref(n, P, D, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((n, D))
    uvi = rng.integers(0, n, (P, 2))
    bad = uvi[:, 0] == uvi[:, 1]
    uvi[bad, 1] = (uvi[bad, 0] + 1) % n
    w = rng.standard_normal(D)
    lat = np.sin(2 * np.pi * x @ w / np.abs(w).sum() + np.pi / 4) + 0.2
    fu = lat[uvi[:, 0]] + 0.05 * rng.standard_normal(P)
    fv = lat[uvi[:, 1]] + 0.05 * rng.standard_normal(P)
    y = np.where(fv > fu, 1.0, -1.0).reshape(-1, 1)
    return x, uvi, y


def test_pref_derivatives_match_reference_semantics(handle):
    uvi, y, f = PREF['k4_uvi'], PREF['k4_y'].astype(float), PREF['k4_f']
    W, g = handle.pref_derivatives(uvi, y, f.reshape(-1))
    oW, og = gppref_oracle.ProbitPrefOracle().derivatives(uvi, y, f)
    assert np.abs(g - og[:, 0]).max() <= 1e-13 * np.abs(og).max()
    assert np.abs(W - oW).max() <= 1e-13 * np.abs(oW).max()
    assert np.abs(np.diag(W) - PREF['k4_Wdiag']).max() <= 1e-13 * np.abs(PREF['k4_Wdiag']).max()
    # accumulate mode differs from the reference exactly where items repeat
    W2, g2 = handle.pref_derivatives(uvi, y, f.reshape(-1), grad_mode=1)
    _, og2 = gppref_oracle.ProbitPrefOracle().derivatives(uvi, y, f, accumulate=True)
    assert np.abs(g2 - og2[:, 0]).max() <= 1e-13 * np.abs(og2).max()
    assert np.abs(g2 - g).max() > 1e-3


def test_pref_laplace_kat3_demo_golden(handle):
    x, uvi, y, lh = PREF['k3_x'], PREF['k3_uvi'], PREF['k3_y'].astype(float), PREF['k3_loghyp']
    handle.set_train(x)
    f, lml, iters, trace, jit = handle.pref_laplace(uvi, y, pref_khyp(lh, 1), delta_f=1e-5)
    assert iters == len(PREF['k3_trace']) == 5
    assert jit == 1e-6
    assert np.abs(f - PREF['k3_f'][:, 0]).max() < 1e-6
    assert abs(lml - float(PREF['k3_lml'])) <= 1e-8 * abs(float(PREF['k3_lml']))
    assert np.abs(trace[:, 1] - PREF['k3_trace'][:, 1]).max() <= 1e-8 * np.abs(PREF['k3_trace'][:, 1]).max()
    assert np.abs(trace[:3, 0] - PREF['k3_trace'][:3, 0]).max() < 1e-8


def test_pref_laplace_kat4_repeated_items_golden(handle):
    x, uvi, y, lh = PREF['k4_x'], PREF['k4_uvi'], PREF['k4_y'].astype(float), PREF['k4_loghyp']
    handle.set_train(x)
    gold_trace = PREF['k4_trace']
    f, lml, iters, trace, _ = handle.pref_laplace(uvi, y, pref_khyp(lh, 3), delta_f=1e-6)
    assert abs(iters - len(gold_trace)) <= 1          # linear convergence: the stop test may tip by one step
    k = min(iters, len(gold_trace))
    assert np.abs(trace[:k, 0] - gold_trace[:k, 0]).max() < 1e-6
    assert np.abs(f - PREF['k4_f'][:, 0]).max() < 2e-6
    assert abs(lml - float(PREF['k4_lml'])) <= 1e-6 * abs(float(PREF['k4_lml']))
    # the same number of iterations as the reference, exactly: mode within 1e-6
    f2, lml2, it2, _, _ = handle.pref_laplace(uvi, y, pref_khyp(lh, 3), delta_f=0.0, max_iter=len(gold_trace))
    assert it2 == len(gold_trace)
    assert np.abs(f2 - PREF['k4_f'][:, 0]).max() < 1e-6
    assert abs(lml2 - float(PREF['k4_lml'])) <= 1e-8 * abs(float(PREF['k4_lml']))


@pytest.mark.parametrize("n,P,D", [(200, 900, 2), (640, 3000, 6)])
def test_pref_laplace_matches_oracle(handle, n, P, D):
    x, uvi, y = make_pref(n, P, D, seed=n)
    lh = np.log([0.5] * D + [1.0, 0.1])
    iters_cap = 25
    of, olml, otrace = gppref_oracle.calc_laplace(x, uvi, y, lh, max_iter=iters_cap, return_trace=True)
    handle.set_train(x)
    f, lml, iters, trace, _ = handle.pref_laplace(uvi, y, pref_khyp(lh, D), delta_f=1e-6, max_iter=iters_cap)
    assert iters == len(otrace)
    assert np.abs(f - of[:, 0]).max() < 1e-6
    assert abs(lml - olml) <= 1e-8 * abs(olml)
    # opt-in Newton mode converges quadratically to the accumulated-gradient mode
    nf, nlml, nit, _, _ = handle.pref_laplace(uvi, y, pref_khyp(lh, D), delta_f=1e-8, max_iter=50, grad_mode=1)
    onf, onlml = gppref_oracle.calc_laplace(x, uvi, y, lh, delta_f=1e-8, max_iter=50, accumulate=True)
    assert nit < 15
    assert np.abs(nf - onf[:, 0]).max() < 1e-6
    assert abs(nlml - onlml) <= 1e-8 * abs(onlml)


def test_gppref_dropin_module(handle):
    from gptest_b200 import GPpref
    x, uvi, y, lh = PREF['k3_x'], PREF['k3_uvi'], PREF['k3_y'], PREF['k3_loghyp']
    gp = GPpref.PreferenceGaussianProcess(x, uvi, y, delta_f=1e-5)
    f, lml = gp.calc_laplace(lh)
    assert f.shape == (40, 1) and isinstance(lml, float)
    assert gp.likelihood.sigma == 1.0                       # GPpref.py:115 quirk
    assert np.abs(f - PREF['k3_f']).max() < 1e-6
    assert abs(gp.calc_nlml(lh) + float(PREF['k3_lml'])) <= 1e-8 * abs(float(PREF['k3_lml']))
    W, g = gp.likelihood.derivatives(uvi, y.astype(float), PREF['k3_f'])
    assert np.abs(W - PREF['k3_W']).max() <= 1e-13 * np.abs(PREF['k3_W']).max()
    assert g.shape == (40, 1) and np.abs(g - PREF['k3_g']).max() <= 1e-13 * np.abs(PREF['k3_g']).max()
    K = gp.kern.K(x)
    assert np.abs(K - gppref_oracle.rbf_ard_K(x, gp.kern.lengthscale, gp.kern.variance)).max() < 1e-14
    assert np.array_equal(np.diag(K), np.full(40, gp.kern.variance))


# ---------------------------------------------------------------------------------------
def make_gpc(n, D, seed):
    from scipy.special import ndtr
    rng = np.random.default_rng(seed)
    x = rng.random((n, D))
    w = rng.standard_normal(D)
    lat = np.sin(2 * np.pi * x @ w / np.abs(w).sum() + np.pi / 4) + 0.2      # GP_classification_demo.py:10-12
    y = np.where(rng.random(n) < ndtr(lat), 1.0, -1.0)                        # :14-21
    z = rng.random((57, D))
    return x, y, z


@pytest.mark.parametrize("n,D,link", [(300, 2, 'probit'), (1000, 4, 'probit'), (500, 3, 'Logit')])
def test_gpc_laplace_and_predict_match_oracle(handle, n, D, link):
    x, y, z = make_gpc(n, D, seed=n + D)
    lh = np.log([0.5] * D + [1.0])
    of, olml, st = gpc_oracle.calc_laplace(x, y, lh, link=link, return_state=True)
    kh = np.concatenate([np.exp(lh[:D]), [np.exp(lh[D]) ** 2]])
    handle.set_train(x)
    f, lml, iters, trace, jit = handle.gpc_laplace(y, kh, link=1 if link == 'Logit' else 0)
    assert iters == st['it'] and jit == st['eps']
    assert np.abs(f - of).max() < 1e-6
    assert abs(lml - olml) <= 1e-8 * abs(olml)
    mu, var, p = handle.gpc_predict(z)
    omu, ovar, op = gpc_oracle.predict(x, y, lh, z, link=link)
    assert np.abs(mu - omu).max() < 1e-7
    assert np.abs(var - ovar).max() < 1e-7
    assert np.abs(p - op).max() < 1e-7


def test_gpc_dropin_module(handle):
    from gptest_b200 import GPc
    x, y, z = make_gpc(260, 1, seed=3)
    y01 = ((y + 1) / 2).astype(int)                                           # {0,1} labels (GPc.py:37)
    gp = GPc.ClassifierGaussianProcess(x, y01)
    lh = np.log([0.3, 1.0])
    f, lml = gp.calc_laplace(lh)
    of, olml = gpc_oracle.calc_laplace(x, y01, lh)
    assert f.shape == (260, 1) and np.abs(f[:, 0] - of).max() < 1e-6
    assert abs(lml - olml) <= 1e-8 * abs(olml)
    mu, var, p = gp.predict(lh, z)
    omu, ovar, op = gpc_oracle.predict(x, y01, lh, z)
    assert np.abs(p - op).max() < 1e-7 and ((p > 0) & (p < 1)).all()
    with pytest.raises(AssertionError):
        GPc.ClassifierGaussianProcess(x, np.full(260, 2))
    assert GPc.ClassifierLikelihood('Logit').link_id == 1 and GPc.ClassifierLikelihood().link_id == 0
    assert abs(GPc.logistic_function(0.0) - 0.5) < 1e-16


# ---- opt-in extensions (SURVEY 8f rank 3): evidence and prediction, against the dense numpy restatement -----
@pytest.mark.parametrize("n,P,D,newton", [(60, 200, 2, True), (300, 1500, 3, True), (200, 700, 2, False)])
def test_pref_evidence_and_prediction(handle, n, P, D, newton):
    x, uvi, y = make_pref(n, P, D, seed=n + P)
    lh = np.log([0.4] * D + [1.2, 0.1])
    handle.set_train(x)
    f, lml, iters, trace, jit = handle.pref_laplace(uvi, y, pref_khyp(lh, D), sigma=1.0, delta_f=1e-9, max_iter=400,
                                                    grad_mode=1 if newton else 0)
    ev = handle.pref_evidence()
    ref = gppref_oracle.laplace_evidence(x, uvi, y, lh, f, sigma=1.0, eps=jit)
    assert abs(ev - ref) <= 1e-8 * max(1.0, abs(ref))
    rng = np.random.default_rng(7)
    za, zb = rng.random((130, D)), rng.random((130, D))
    mu, var = handle.pref_predict(za)
    rmu, rvar = gppref_oracle.predict_latent(x, uvi, y, lh, f, za, eps=jit)
    # k** - k*'K^-1 k* cancels to ~1e-6 * sf2 with the 1e-6 jitter: absolute tolerance on the prior scale
    assert np.abs(mu - rmu).max() <= 1e-7 * max(1.0, np.abs(rmu).max())
    assert np.abs(var - rvar).max() <= 1e-7
    dmu, dvar, p = handle.pref_predict(za, zb)
    rdmu, rdvar, rp = gppref_oracle.predict_latent(x, uvi, y, lh, f, za, zb, eps=jit)
    assert np.abs(dmu - rdmu).max() <= 1e-7 * max(1.0, np.abs(rdmu).max())
    assert np.abs(dvar - rdvar).max() <= 1e-7
    assert np.abs(p - rp).max() <= 1e-7 and ((p > 0) & (p < 1)).all()
    # symmetry: swapping the items flips the mean and the probability
    dmu2, dvar2, p2 = handle.pref_predict(zb, za)
    assert np.abs(dmu + dmu2).max() < 1e-9 and np.abs(p + p2 - 1).max() < 1e-9
    # training items predict their own mode
    mu_t, var_t = handle.pref_predict(x[:50])
    assert np.abs(mu_t - f[:50]).max() < 1e-5


def test_pref_state_is_invalidated_by_other_calls(handle):
    from gptest_b200._lib import GpbError
    x, uvi, y = make_pref(50, 120, 2, seed=1)
    lh = np.log([0.4, 0.4, 1.2, 0.1])
    handle.set_train(x)
    handle.pref_laplace(uvi, y, pref_khyp(lh, 2), sigma=1.0, delta_f=1e-6, max_iter=100)
    handle.pref_evidence()
    handle.pref_predict(x[:3])                     # the state survives its own readers
    handle.kxx(np.array([0.4, 0.4, 1.0, 0.0]))     # ... but not a call that uses the work space
    with pytest.raises(GpbError, match='gpb_pref_laplace first'):
        handle.pref_evidence()
    yc = np.where(np.arange(50) % 2 == 0, 1.0, -1.0)
    handle.gpc_laplace(yc, np.array([0.4, 0.4, 1.0]))
    handle.gpc_predict(x[:3])
    handle.gpc_predict(x[:3])
    handle.kxx(np.array([0.4, 0.4, 1.0, 0.0]))
    with pytest.raises(GpbError, match='gpb_gpc_laplace first'):
        handle.gpc_predict(x[:3])
    # one state per handle: a fit of the other kind on the same n replaces it
    handle.pref_laplace(uvi, y, pref_khyp(lh, 2), sigma=1.0, delta_f=1e-6, max_iter=100, grad_mode=1)
    handle.pref_evidence()                         # the factor of K^-1 + W is in the work space
    handle.gpc_laplace(yc, np.array([0.4, 0.4, 1.0]))
    for call in (handle.pref_evidence, lambda: handle.pref_predict(x[:3]), handle.pref_evidence_grad):
        with pytest.raises(GpbError, match='gpb_pref_laplace first'):
            call()
    handle.gpc_laplace(yc, np.array([0.4, 0.4, 1.0]))
    handle.pref_laplace(uvi, y, pref_khyp(lh, 2), sigma=1.0, delta_f=1e-6, max_iter=100, grad_mode=1)
    for call in (lambda: handle.gpc_predict(x[:3]), handle.gpc_evidence_grad):
        with pytest.raises(GpbError, match='gpb_gpc_laplace first'):
            call()


def test_gppref_dropin_extensions(handle):
    from gptest_b200 import GPpref
    x, uvi, y, lh = PREF['k3_x'], PREF['k3_uvi'], PREF['k3_y'], PREF['k3_loghyp']
    gp = GPpref.PreferenceGaussianProcess(x, uvi, y, delta_f=1e-9, newton=True)
    f, lml = gp.calc_laplace(lh)
    ev = gp.laplace_evidence()
    ref = gppref_oracle.laplace_evidence(x, uvi, y, lh, f, eps=gp.jitter)
    assert abs(ev - ref) <= 1e-8 * max(1.0, abs(ref))
    mu, var, p = gp.predict_preference(x[:5], x[5:10])
    assert p.shape == (5,) and np.all(var > -1e-9)


@pytest.mark.parametrize("n,P", [(40, 120), (77, 300)])
def test_pref_log_marginal_on_device(handle, n, P):
    """PrefProbit.log_marginal (GPpref.py:90-94) with caller-supplied iK / logdetK, odd and even n."""
    from gptest_b200 import GPpref
    x, uvi, y = make_pref(n, P, 3, seed=n)
    rng = np.random.default_rng(n)
    f = 0.3 * rng.standard_normal((n, 1))
    K = gppref_oracle.rbf_ard_K(x, np.array([0.5, 0.5, 0.5]), 1.3) + 1e-6 * np.eye(n)
    L = np.linalg.cholesky(K)
    iK = np.linalg.inv(K)
    logdetK = np.sum(np.log(np.diag(L)))                       # GPpref.py:131
    for sigma in (1.0, 0.4):
        ref = gppref_oracle.ProbitPrefOracle(sigma).log_marginal(uvi, y, f, iK, logdetK)
        lik = GPpref.PrefProbit(sigma)
        got = lik.log_marginal(uvi, y, f, iK, logdetK)
        assert isinstance(got, float) and abs(got - ref) <= 1e-10 * max(1.0, abs(ref))


def test_laplace_loops_on_the_callers_default_stream():
    """A caller may hand the library the legacy default stream (torch.cuda.current_stream() is that one unless the
    caller made a stream): it cannot be captured into a graph, so the device loop runs on a stream of the handle's own,
    ordered after the caller's.  Same numbers as on the handle's stream."""
    from gptest_b200 import _lib
    h = _lib.Handle(0)
    try:
        h.set_stream(0)
        x, uvi, y, lh = PREF['k3_x'], PREF['k3_uvi'], PREF['k3_y'].astype(float), PREF['k3_loghyp']
        h.set_train(x)
        f, lml, iters, trace, jit = h.pref_laplace(uvi, y, pref_khyp(lh, 1), delta_f=1e-5)
        assert iters == 5 and np.abs(f - PREF['k3_f'][:, 0]).max() < 1e-6
        assert abs(lml - float(PREF['k3_lml'])) <= 1e-8 * abs(float(PREF['k3_lml']))
        xc, yc, zc = make_gpc(300, 2, seed=302)
        lhc = np.log([0.5, 0.5, 1.0])
        of, olml, st = gpc_oracle.calc_laplace(xc, yc, lhc, return_state=True)
        h.set_train(xc)
        fc, lmlc, itc, _, _ = h.gpc_laplace(yc, np.array([0.5, 0.5, 1.0]))
        assert itc == st['it'] and np.abs(fc - of).max() < 1e-6 and abs(lmlc - olml) <= 1e-8 * abs(olml)
    finally:
        h.close()
