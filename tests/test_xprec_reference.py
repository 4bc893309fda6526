"""The extended-precision reference (tests/_xprec.py) checked on the CPU, and the CPU model of the device's order of
operations held to the envelope the GPU tests use.

  * the reference is exact where exact arithmetic is representable, and at least 100x closer than float64 LAPACK to
    a 50-digit mpmath computation up to cond(K) ~ 1e12, the largest condition number tests/test_gpu_conditioning.py uses;
  * the design (inverted 32-blocks, TRSM as a product with the inverse, z = W r) against the envelope
    |emulation - truth| <= 10 |LAPACK - truth| + 16 n u |value| and backward error <= 4 n u: inside up to cond ~ 1e8,
    outside on some inputs from there on, as the device; a variant that forms the inverse the unstable way,
    W = L^T (L L^T)^-1, leaves it far on F1 and stays inside on the control - so the envelope has teeth.
"""
import numpy as np
import pytest

from oracle import gpr_oracle
from tests import _xprec as xp

pytestmark = pytest.mark.skipif(np.finfo(np.longdouble).eps > 1e-18,
                                reason='np.longdouble is not wider than float64 on this platform (eps %g): '
                                       'the extended-precision reference needs 80-bit or 128-bit long double'
                                       % np.finfo(np.longdouble).eps)


def f1(n, sn, seed=1, ell=0.3):
    """F1: squared exponential on dense 1-D inputs in [0, 1]; cond(K) ~ 1.5e4 / sn^2 ... at n = 256."""
    rng = np.random.default_rng(seed)
    x = rng.random((n, 1))
    y = np.sin(6 * x[:, 0]) + 0.1 * rng.standard_normal(n)
    return gpr_oracle.kxx(np.log([ell, 1.0, sn]), x), x, y


def f2(n, sn, seed=1):
    """F2: squared exponential, D = 8, l = 0.5: cond(K) saturates near 1e3..1e4 whatever sn (the control)."""
    rng = np.random.default_rng(seed)
    x = rng.random((n, 8))
    y = np.sin(x.sum(1)) + 0.1 * rng.standard_normal(n)
    return gpr_oracle.kxx(np.log([0.5] * 8 + [1.0, sn]), x), x, y


# ---------------------------------------------------------------------------------------------------------------------
# the reference itself
# ---------------------------------------------------------------------------------------------------------------------
def test_integer_factor_is_reproduced_exactly():
    """A = L L^T with a small-integer L is exact in float64, every pivot is a perfect square and every division exact:
    the long-double Cholesky must return L itself, and the solves the exact rational answer."""
    rng = np.random.default_rng(0)
    n = 40
    L = np.tril(rng.integers(-3, 4, (n, n)), -1).astype(np.float64)
    L[np.diag_indices(n)] = rng.integers(1, 4, n)
    A = L @ L.T
    assert np.abs(A).max() < 2 ** 40                   # exact in float64 and in every intermediate
    E = xp.Exact(A)
    assert np.array_equal(E.L.astype(np.float64), L)
    assert np.array_equal(E.L, np.tril(E.L))
    b = L @ np.arange(1.0, n + 1)                       # L z = b has the integer solution 1..n
    assert np.array_equal(E.z(b).astype(np.float64), np.arange(1.0, n + 1))
    assert xp.llt_residual(E.L, A) == 0.0
    W = xp.tril_inv_ld(E.L)                             # thirds and halves: not exact, but long-double close
    assert np.array_equal(W, np.tril(W))
    assert float(np.abs(W @ E.L - np.eye(n)).max()) < 1e3 * xp.ld_eps() * float(np.abs(W).max())


def _mp_truth(K, y, Kxz, sf2):
    import mpmath as mp
    n = len(K)
    A = mp.matrix(K.tolist())
    L = mp.cholesky(A)
    z = [mp.mpf(0)] * n
    for i in range(n):
        z[i] = (mp.mpf(y[i]) - mp.fsum(L[i, k] * z[k] for k in range(i))) / L[i, i]
    nlml = mp.fsum(v * v for v in z) / 2 + mp.fsum(mp.log(L[i, i]) for i in range(n)) + n * mp.log(2 * mp.pi) / 2
    alpha = [mp.mpf(0)] * n
    for i in range(n - 1, -1, -1):
        alpha[i] = (z[i] - mp.fsum(L[k, i] * alpha[k] for k in range(i + 1, n))) / L[i, i]
    m = Kxz.shape[1]
    mean = [mp.fsum(mp.mpf(Kxz[k, j]) * alpha[k] for k in range(n)) for j in range(m)]
    var = []
    for j in range(m):
        v = [mp.mpf(0)] * n
        for i in range(n):
            v[i] = (mp.mpf(Kxz[i, j]) - mp.fsum(L[i, k] * v[k] for k in range(i))) / L[i, i]
        var.append(mp.mpf(sf2) - mp.fsum(t * t for t in v))
    Lf = np.array([[float(L[i, j]) if j <= i else 0.0 for j in range(n)] for i in range(n)])
    return L, nlml, mean, var, Lf


@pytest.mark.parametrize('sn', [5e-5, 5e-6], ids=['cond1e10', 'cond1e12'])
def test_reference_is_100x_closer_to_mpmath_than_lapack(sn):
    """C3: at the largest condition numbers the GPU tests use, the long-double reference must be at least 100 times
    more accurate than float64 LAPACK - otherwise 'gpu vs reference' would measure the reference."""
    import mpmath as mp
    mp.mp.dps = 50
    n = 48
    rng = np.random.default_rng(3)
    x = np.sort(rng.random(n))
    y = np.sin(6 * x) + 0.1 * rng.standard_normal(n)
    z = rng.random(6)
    lh = np.log([0.3, 1.0, sn])
    K = gpr_oracle.kxx(lh, x)
    Kxz = gpr_oracle.kxz(lh, x, z)
    cond = np.linalg.cond(K)
    assert (5e9 if sn == 5e-5 else 5e11) < cond < (5e10 if sn == 5e-5 else 5e12), cond
    Lmp, nl_mp, mean_mp, var_mp, _ = _mp_truth(K, y, Kxz, 1.0)
    E, P = xp.Exact(K), xp.Lapack(K)

    def err(v, ref):
        return float(mp.mpf(abs(mp.mpf(str(v)) - ref)))     # str(): the long double's full digits

    e_ld, e_lp = err(E.nlml(y), nl_mp), err(P.nlml(y), nl_mp)
    assert e_ld * 100 <= e_lp, ('NLML', e_ld, e_lp)
    eL_ld = max(err(E.L[i, j], Lmp[i, j]) for i in range(n) for j in range(i + 1))
    eL_lp = max(err(P.L[i, j], Lmp[i, j]) for i in range(n) for j in range(i + 1))
    assert eL_ld * 100 <= eL_lp, ('L', eL_ld, eL_lp)
    m_ld, v_ld = E.predict(y, Kxz, 1.0)
    m_lp, v_lp = P.predict(y, Kxz, 1.0)
    em_ld = max(err(a, b) for a, b in zip(m_ld, mean_mp))
    em_lp = max(err(a, b) for a, b in zip(m_lp, mean_mp))
    assert em_ld * 100 <= em_lp, ('mean', em_ld, em_lp)
    ev_ld = max(err(a, b) for a, b in zip(v_ld, var_mp))
    ev_lp = max(err(a, b) for a, b in zip(v_lp, var_mp))
    assert ev_ld * 100 <= ev_lp or ev_lp < 1e-15, ('variance', ev_ld, ev_lp)


def test_reference_gradient_matches_central_differences():
    """The long-double SE gradient is the derivative of the long-double NLML (central differences of the float64 K
    assembled at shifted log hyper-parameters), at a moderate conditioning where differencing resolves it."""
    rng = np.random.default_rng(4)
    n, d = 60, 2
    x = rng.random((n, d))
    y = np.sin(x @ [3.0, -2.0]) + 0.1 * rng.standard_normal(n)
    lh = np.log([0.4, 0.6, 1.1, 0.05])
    ell, sf2, sn2 = gpr_oracle.split_hyp(lh)
    khyp = np.r_[ell, sf2, sn2]
    K = gpr_oracle.kxx(lh, x)
    g = xp.Exact(K).se_grad(x, y, khyp).astype(np.float64)
    h = 1e-5
    fd = np.empty(d + 2)
    for k in range(d + 2):
        e = np.zeros(d + 2)
        e[k] = h
        fp = float(xp.Exact(gpr_oracle.kxx(lh + e, x)).nlml(y))
        fm = float(xp.Exact(gpr_oracle.kxx(lh - e, x)).nlml(y))
        fd[k] = (fp - fm) / (2 * h)
    assert np.abs(g - fd).max() <= 1e-6 * np.abs(g).max(), (g, fd)
    gl = xp.Lapack(K).se_grad(x, y, khyp)
    assert np.abs(g - gl).max() <= 1e-10 * np.abs(g).max()
    assert np.abs(g - gpr_oracle.nlml_grad(lh, x, y)).max() <= 1e-10 * np.abs(g).max()


# ---------------------------------------------------------------------------------------------------------------------
# the design's order of operations, modelled on the CPU
# ---------------------------------------------------------------------------------------------------------------------
def _envelope(K, y, **kw):
    n = len(K)
    truth = xp.Exact(K).nlml(y)
    try:
        val, L = xp.emulate_nlml(K, y, **kw)
        bw = xp.llt_residual(L, K)
    except np.linalg.LinAlgError:                     # the model broke down: outside any envelope
        val, bw = np.nan, np.inf
    ok, ratio, _, _ = xp.forward_check(val, xp.lapack_samples(K, lambda P, p: P.nlml(y[p])), truth, n,
                                       abs(float(truth)))
    return ok and bw <= xp.backward_bound(n), ratio, bw


@pytest.mark.parametrize('fam,sn,inside', [('F1', 1e-2, True), ('F1', 1e-4, False), ('F2', 1e-2, True),
                                           ('F2', 1e-4, True)])
def test_design_order_against_the_envelope(fam, sn, inside):
    """The design's order is inside the envelope at cond ~ 1e6 and on the control, and outside it at cond ~ 1e10
    (ratio ~ 15 against the median LAPACK error; its backward error stays under 4 n u there)."""
    K, _, y = (f1 if fam == 'F1' else f2)(256, sn)
    ok, ratio, bw = _envelope(K, y)
    assert ok == inside, 'emulation / LAPACK NLML error ratio %.3g, backward error %.3g (bound %.3g)' % (
        ratio, bw, xp.backward_bound(256))


def test_unstable_inverse_fails_the_envelope_only_when_ill_conditioned():
    """W = L^T (L L^T)^-1 squares cond(L_kk): harmless on the well-conditioned control F2, far outside the envelope on
    F1 at sn = 1e-4 (cond ~ 1e10).  A kernel defect of that kind is what the GPU criteria must catch."""
    K, _, y = f2(256, 1e-4)
    ok, ratio, bw = _envelope(K, y, unstable_w=True)
    assert ok, 'F2: ratio %.3g, backward error %.3g' % (ratio, bw)
    K, _, y = f1(256, 1e-4)
    ok, ratio, bw = _envelope(K, y, unstable_w=True)
    assert not ok, 'F1 sn=1e-4: the unstable inverse stayed inside the envelope (ratio %.3g)' % ratio
    assert not ratio <= 100                           # nan (breakdown) or far outside, not a near miss


# The F1 value checks the B200 leaves outside C1 (tests/test_gpu_conditioning.py KNOWN, device ratio in the comment),
# and whether the CPU model of the design leaves it too on the same inputs (numpy's K: the device's differs by ulps).
DEVICE_OUTSIDE = [                 # (n, sn, the model is outside as well)
    (128, 1e-4, True),             # device 47
    (128, 1e-5, False),            # device 56
    (200, 1e-3, True),             # device 16
    (200, 1e-4, True),             # device 10
    (200, 1e-5, True),             # device 736
    (384, 1e-5, True),             # device 22
    (512, 1e-3, False),            # device 12
    (512, 1e-4, True),             # device 103
    (512, 1e-5, True),             # device 118
    (1000, 1e-4, False),           # device 24
]


@pytest.mark.parametrize('n,sn,design', DEVICE_OUTSIDE)
def test_design_model_on_the_cases_the_device_misses(n, sn, design):
    """Classifies each NLML case the device misses: where the model of the design's order misses too, the inverse-based
    solves explain it; where the model stays inside, the device's excess is not explained by the design (DESIGN.md 9)."""
    X, y, _, kh, _ = xp.gp_inputs('F1', n, sn)
    K = gpr_oracle.kxx(np.log([kh[0], 1.0, sn]), X)
    truth = xp.Exact(K).nlml(y)
    val, _ = xp.emulate_nlml(K, y)
    ok, ratio, _, _ = xp.forward_check(val, xp.lapack_samples(K, lambda P, p: P.nlml(y[p])), truth, n,
                                       abs(float(truth)))
    assert ok != design, 'model/LAPACK NLML error ratio %.3g' % ratio
