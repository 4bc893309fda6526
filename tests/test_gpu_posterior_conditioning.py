"""Joint posterior covariance and posterior samples (gpb_gpr_predict_full, gpb_gpr_sample; posterior.cu, DESIGN.md 4.8)
against an extended-precision reference across the conditioning range.

The oracle parity test (tests/test_gpu_gpr_posterior.py) holds Sigma* to 1e-9 sf2 at sn^2 = 0.04, where a product that
drops a k-slab of V still passes.  Here, as in tests/test_gpu_conditioning.py, every reference is computed on the
device's OWN matrices (K and Kxz after set_train(X, y), Kzz after set_train(Z)) in long double (tests/_xprec.py), and
each device result is held to float64 LAPACK's accuracy on the same matrices:

  P1  C1 on the whole m x m Sigma* of predict_full: |gpu - truth| <= 10 |lapack - truth| + 16 n u sf2 (max norms;
      |lapack - truth| the median over K and 4 symmetric permutations of it); the message splits the diagonal and the
      off-diagonal errors
  P2  Sigma* exactly symmetric, two calls the same bits, Sigma* independent of the mean, and fz of predict_full equal to
      gpr_predict's bit for bit with mean = 0.7
  P3  P1 under split_tiles = 0 (128 x 128 CTA tiles: the other instantiation of the DMMA kernel)
  S1  the sampler's factor L*: with y = 0, fz = 0 exactly and the samples are D = E L*^T exactly; L* is recovered by
      least squares from S = 4 m draws (xp.recover_factor, tests/test_xprec_reference.py calibrates it), its strict
      upper triangle must be <= 1e-14 max|L*|, and C2 (backward error <= 4 m u) holds against Sigma* + eps I with the
      device's own Sigma* and returned jitter eps
  S2  the jitter rung: with delta = 64 m u max|Sigma* + eps I|, Sigma* + (eps + delta) I factors in long double, and
      when eps > 0, Sigma* + (eps_prev - delta) I does not (eps_prev the rung below): the device neither accepts an
      indefinite matrix nor over-jitters.  Where the sampler's factor leaves C2, gpb_potrf_lower of the same matrix is
      measured beside it, and gpr_predict's variance beside Sigma*: that tells the factorisation's and V's share
  S3  samples(y, mean = 0.7) = fz + samples(y = 0) bit for bit (the single add of sample_finish_kernel)

Cases (family, n, sn) of tests/_xprec.gp_inputs, F5 being Matern 5/2; the number of test points m cycles through
1, 2, 33, 65, 129, 257, 384 (a single Philox pair; the mirror's 32-tiles; the 64-padded test rows against the
128-padded Sigma*; a V region shorter than the product's tiles; several tiles), and noisy alternates.  The test
points mix the three kinds of xp.posterior_points: inside the data, on training points, outside.

A check outside its criterion on the B200 is listed in KNOWN with its measured figure and held to twice it (DESIGN.md
9).  Every check of a test runs before the test reports.  GPB_POSTERIOR_TABLE=<file> writes the table of all checks
(profiles/r06_posterior_conditioning.txt).
"""
import contextlib
import os

import numpy as np
import pytest

import bench_configs as cfg
from tests import _xprec as xp
from tests._posterior_oracle import philox_normals

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(np.finfo(np.longdouble).eps > 1e-18,
                                 reason='np.longdouble is not wider than float64 here: no extended-precision reference')]

FAMILY_CASES = ([('F1', n, sn) for n in (128, 200, 384) for sn in (1e-1, 1e-3, 1e-5)]
                + [('F1', 1000, sn) for sn in (1e-1, 1e-3, 1e-4)]
                + [('F2', n, sn) for n in (128, 512) for sn in (1e-1, 1e-3)]
                + [(fam, n, 1e-3) for fam in ('F3', 'F5') for n in (200, 1000)])
MS = [1, 2, 33, 65, 129, 257, 384]
CASES = [(fam, n, sn, MS[i % len(MS)], i % 2 == 1) for i, (fam, n, sn) in enumerate(FAMILY_CASES)]
SAMPLER_CASES = [c for c in CASES if c[3] in (33, 129, 257)]
SPLIT_CASES = [c for c in CASES if (c[0], c[1], c[2]) in (('F1', 384, 1e-5), ('F1', 1000, 1e-4), ('F2', 512, 1e-3),
                                                          ('F5', 1000, 1e-3))]
LADDER = np.array([0.0, 1e-12, 1e-11, 1e-10, 1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1, 1.0])  # posterior.cu
SEED = 0x0123_4567_89ab_cdef
TABLE = []

# Measured on the B200 (profiles/r06_posterior_conditioning.txt): checks outside their criterion, keyed (check, family,
# n, sn), with the measured gpu/LAPACK ratio (backward-error checks: the backward error in units of m u; the jitter
# rung: rungs over).  Each is held to twice its figure.  Sigma* leaves C1 exactly where gpr_predict's variance at the
# same points does: the excess is V's (the factorisation with the test rows riding along, DESIGN.md 9), not the
# product's.  The sampler's factor leaves C2 where gpb_potrf_lower of the same Sigma* + eps I does too.
KNOWN = {
    ('Sigma*', 'F1', 128, 1e-05): 28,
    ('Sigma*', 'F1', 200, 0.001): 31.2,
    ('Sigma*', 'F1', 200, 1e-05): 285,
    ('Sigma*', 'F1', 1000, 0.0001): 77.4,
    ('Sigma* split_tiles=0', 'F1', 1000, 0.0001): 77.4,
    ('predict variance', 'F1', 128, 1e-05): 28,
    ('predict variance', 'F1', 200, 0.001): 31.2,
    ('predict variance', 'F1', 200, 1e-05): 285,
    ('predict variance', 'F1', 1000, 0.0001): 77.4,
    ('sampler backward', 'F1', 128, 1e-05): 69.1,
    ('sampler backward', 'F1', 200, 0.001): 135,
    ('sampler backward', 'F1', 200, 1e-05): 7.18,
    ('sampler backward', 'F1', 1000, 0.0001): 7.34,
    ('sampler backward', 'F5', 200, 0.001): 6,
    ('potrf of Sigma*+epsI', 'F1', 128, 1e-05): 69.2,
    ('potrf of Sigma*+epsI', 'F1', 200, 0.001): 135,
    ('potrf of Sigma*+epsI', 'F1', 200, 1e-05): 7.18,
    ('potrf of Sigma*+epsI', 'F1', 1000, 0.0001): 7.34,
    ('potrf of Sigma*+epsI', 'F5', 200, 0.001): 6.01,
    ('jitter rung', 'F1', 200, 0.001): 1,
}
RESULTS = []


@pytest.fixture(autouse=True)
def _results():
    RESULTS.clear()
    yield


@contextlib.contextmanager
def split_tiles(handle, value):
    try:
        handle.set_option('split_tiles', value)
        yield
    finally:
        handle.set_option('split_tiles', 1)


class Case:
    """One posterior problem: the device's K, Kxz and Kzz, and the long-double and LAPACK Sigma* on them (once)."""

    def __init__(self, handle, fam, n, sn, m, noisy, X, y, Z, khyp, kind):
        self.fam, self.n, self.sn, self.m, self.noisy = fam, n, sn, m, noisy
        self.X, self.y, self.Z, self.khyp, self.kind = X, y, Z, khyp, kind
        self.sf2 = khyp[-2]
        handle.set_train(Z)                             # Kzz: the noise only on the predictive of observations
        self.Kzz = handle.kxx(khyp if noisy else np.r_[khyp[:-1], 0.0], kind=kind)
        self.train(handle)
        self.K = handle.kxx(khyp, kind=kind)
        self.Kxz = handle.kxz(khyp, Z, kind=kind)
        ev = np.linalg.eigvalsh(self.K)
        self.cond = ev[-1] / ev[0] if ev[0] > 0 else np.inf
        self._memo = {}

    def memo(self, key, f):
        if key not in self._memo:
            self._memo[key] = f()
        return self._memo[key]

    def sigma(self):
        """(truth, LAPACK samples) of Sigma*."""
        return (self.memo('E', lambda: xp.Exact(self.K).posterior_cov(self.Kxz, self.Kzz)),
                self.memo('P', lambda: xp.lapack_samples(self.K, lambda P, p: P.posterior_cov(self.Kxz[p], self.Kzz))))

    def train(self, handle, y=None):
        handle.set_train(self.X, self.y if y is None else y)

    def label(self):
        return '%s n=%d sn=%.0e m=%d %s' % (self.fam, self.n, self.sn, self.m, 'noisy' if self.noisy else 'latent')


@pytest.fixture(scope='module')
def cases(handle):
    """case(fam, n, sn, m, noisy): built once per module."""
    cache = {}

    def get(fam, n, sn, m, noisy):
        key = (fam, n, sn, m, noisy)
        if key not in cache:
            X, y, _, kh, kind = xp.gp_inputs(fam, n, sn)
            cache[key] = Case(handle, fam, n, sn, m, noisy, X, y, xp.posterior_points(X, m, seed=n + m), kh, kind)
        return cache[key]

    yield get
    path = os.environ.get('GPB_POSTERIOR_TABLE')
    if path:
        write_table(path)


def record(path, case, ok, known, status, ratio, eg, el, msg):
    """One row of the table and one entry of RESULTS; a KNOWN check is held to twice its measured figure."""
    if known is not None:
        status = 'known %.3g' % known
        ok = ratio <= 2 * known
    TABLE.append((path, case, ratio, eg, el, status if ok else 'FAIL (' + status + ')'))
    RESULTS.append((ok, '%s, %s (cond %.1e): %s%s' % (path, case.label(), case.cond, msg,
                                                      '' if known is None else ', measured before %.3g' % known)))


def check_sigma(path, case, S):
    """P1 on the m x m Sigma* of the device."""
    truth, lap = case.sigma()
    ok, ratio, eg, el = xp.forward_check(S, lap, truth, case.n, case.sf2)
    err = np.abs(np.asarray(S, dtype=xp.LD) - truth).astype(np.float64)
    off = ~np.eye(case.m, dtype=bool)
    msg = ('gpu/LAPACK error ratio %.3g (gpu %.3g: diagonal %.3g, off-diagonal %.3g; LAPACK %.3g; floor %.3g)' % (
        ratio, eg, np.diagonal(err).max(), err[off].max() if case.m > 1 else 0.0, el, 16 * case.n * xp.U * case.sf2))
    record(path, case, ok, KNOWN.get((path, case.fam, case.n, case.sn)), 'pass' if ok else 'FAIL', ratio, eg, el, msg)


def settle():
    """Every check of the test has run: report all that failed."""
    bad = [m for ok, m in RESULTS if not ok]
    assert not bad, '\n'.join(bad)


def write_table(path):
    import torch
    lines = ['# tests/test_gpu_posterior_conditioning.py on %s: device error / float64 LAPACK error, both against the'
             % torch.cuda.get_device_name(0),
             '# long-double reference on the device\'s own K, Kxz and Kzz (C1 passes at ratio <= 10 or under the floor',
             '# 16 n u sf2).  LAPACK error: median over K and 4 symmetric permutations of it.  "known r": held to 2 r.',
             '# backward rows (the sampler\'s recovered factor, gpb_potrf_lower on the same A = Sigma* + eps I):',
             '# max|LL^T - A|/max|A| in units of m u for the device and for numpy\'s Cholesky of A (C2: device <= 4).',
             '# jitter rows: ratio = rungs over the lowest that factors in long double with a margin delta, err gpu =',
             '# delta / sf2 = 64 m u max|Sigma* + eps I| / sf2, err lapack = the device\'s eps / sf2.',
             '%-26s %-5s %5s %-7s %4s %-6s %9s %10s %10s %9s %s' % ('check', 'fam', 'n', 'sn', 'm', 'kind', 'cond(K)',
                                                                 'err gpu', 'err lapack', 'ratio', 'status')]
    for path_, c, ratio, eg, el, status in TABLE:
        lines.append('%-26s %-5s %5d %-7.0e %4d %-6s %9.1e %10.3g %10.3g %9.3g %s' % (
            path_, c.fam, c.n, c.sn, c.m, 'noisy' if c.noisy else 'latent', c.cond, eg, el, ratio, status))
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, 'w') as f:
        f.write('\n'.join(lines) + '\n')


def ids(params):
    return ['%s-%d-%g-m%d-%s' % (f, n, sn, m, 'noisy' if nz else 'latent') for f, n, sn, m, nz in params]


# ---------------------------------------------------------------------------------------------------------------------
# Sigma*
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('fam,n,sn,m,noisy', CASES, ids=ids(CASES))
def test_predict_full(handle, cases, fam, n, sn, m, noisy):
    """P1 and P2."""
    c = cases(fam, n, sn, m, noisy)
    c.train(handle)
    fz, S = handle.gpr_predict_full(c.khyp, c.Z, kind=c.kind, noisy=noisy)
    check_sigma('Sigma*', c, S)
    fz2, S2 = handle.gpr_predict_full(c.khyp, c.Z, kind=c.kind, noisy=noisy)
    RESULTS.append((np.array_equal(S, S.T), 'Sigma* of %s is not exactly symmetric' % c.label()))
    RESULTS.append((np.array_equal(S, S2) and np.array_equal(fz, fz2), 'two calls differ on %s' % c.label()))
    fzm, Sm = handle.gpr_predict_full(c.khyp, c.Z, mean=0.7, kind=c.kind, noisy=noisy)
    mu, var = handle.gpr_predict(c.khyp, c.Z, mean=0.7, kind=c.kind)
    RESULTS.append((np.array_equal(fzm, mu), 'fz of predict_full and gpr_predict differ with mean 0.7 on %s: %.3g' % (
        c.label(), np.abs(fzm - mu).max())))
    RESULTS.append((np.array_equal(Sm, S), 'Sigma* depends on the mean on %s' % c.label()))
    # gpr_predict's variance at the same points shares V with Sigma*: an excess of both comes from V, not the product
    truth, lap = c.sigma()
    sn2 = c.khyp[-1] if noisy else 0.0
    ok, ratio, eg, el = xp.forward_check(var, [np.diagonal(v) - sn2 for v in lap], np.diagonal(truth) - xp.LD(sn2),
                                         c.n, c.sf2)
    record('predict variance', c, ok, KNOWN.get(('predict variance', fam, n, sn)), 'pass' if ok else 'FAIL',
           ratio, eg, el, 'gpu/LAPACK error ratio %.3g (gpu %.3g, LAPACK %.3g)' % (ratio, eg, el))
    settle()


@pytest.mark.parametrize('fam,n,sn,m,noisy', SPLIT_CASES, ids=ids(SPLIT_CASES))
def test_predict_full_split_tiles_0(handle, cases, fam, n, sn, m, noisy):
    """P3: the product of Sigma* on 128 x 128 CTA tiles."""
    c = cases(fam, n, sn, m, noisy)
    c.train(handle)
    with split_tiles(handle, 0):
        _, S = handle.gpr_predict_full(c.khyp, c.Z, kind=c.kind, noisy=noisy)
    check_sigma('Sigma* split_tiles=0', c, S)
    settle()


# ---------------------------------------------------------------------------------------------------------------------
# the sampler
# ---------------------------------------------------------------------------------------------------------------------
def check_jitter(handle, case, S, eps):
    """S2 on the device's Sigma* and returned jitter.  Over-jittering is measured in rungs: the ratio is the number of
    rungs between the device's and the lowest one at which Sigma* + (rung - delta) I factors in long double."""
    m, sf2 = case.m, case.sf2
    rung = np.flatnonzero(LADDER * sf2 == eps)
    eye = np.eye(m)
    A = S + eps * eye
    delta = 64 * m * xp.U * float(np.abs(A).max())
    bad, over = [], 0
    if len(rung) != 1:
        bad.append('jitter %r is not a rung of the ladder' % eps)
    elif not xp.ld_factors(S + (eps + delta) * eye):
        bad.append('Sigma* + (eps + delta) I does not factor: the device accepted an indefinite matrix')
    else:
        k = rung[0]
        while k - over > 0 and xp.ld_factors(S + (LADDER[k - over - 1] * sf2 - delta) * eye):
            over += 1
    msg = 'jitter %.3g sf2, delta %.3g sf2' % (eps / sf2, delta / sf2)
    if over:
        try:
            handle.potrf(S + LADDER[rung[0] - 1] * sf2 * eye)
            dev = 'factors'
        except np.linalg.LinAlgError:
            dev = 'fails too'
        msg += ': Sigma* + (eps_prev - delta) I factors, the device over-jittered by %d rung(s) (gpb_potrf_lower of ' \
               'Sigma* + eps_prev I %s)' % (over, dev)
    known = KNOWN.get(('jitter rung', case.fam, case.n, case.sn))
    ok = not bad and (over == 0 if known is None else over <= 2 * known)
    status = 'pass (eps %.0e sf2)' % (eps / sf2) if not bad and over == 0 else 'FAIL'
    record('jitter rung', case, ok, known, status, over, delta / sf2, eps / sf2, msg + (': ' + bad[0] if bad else ''))


@pytest.mark.parametrize('fam,n,sn,m,noisy', SAMPLER_CASES, ids=ids(SAMPLER_CASES))
def test_sampler_factor(handle, cases, fam, n, sn, m, noisy):
    """S1 and S2, with y = 0: the samples are D = E L*^T exactly."""
    c = cases(fam, n, sn, m, noisy)
    c.train(handle, y=np.zeros(n))
    fz, S = handle.gpr_predict_full(c.khyp, c.Z, kind=c.kind, noisy=noisy)
    D, eps = handle.gpr_sample(c.khyp, c.Z, 4 * m, seed=SEED, kind=c.kind, noisy=noisy)
    c.train(handle)
    RESULTS.append((not fz.any(), 'fz is not exactly 0 with y = 0 on %s' % c.label()))
    L = xp.recover_factor(philox_normals(SEED, 4 * m, m), D)
    upper = float(np.abs(np.triu(L, 1)).max() / np.abs(L).max())
    RESULTS.append((upper <= 1e-14, 'the recovered factor of %s has a strict upper triangle of %.3g max|L|' % (
        c.label(), upper)))
    A = S + eps * np.eye(m)
    bw = xp.llt_residual(L, A) / (m * xp.U)
    try:
        bl = xp.llt_residual(np.linalg.cholesky(A), A) / (m * xp.U)
    except np.linalg.LinAlgError:
        bl = np.nan
    # the device's gpb_potrf_lower on the same matrix: the sampler adds nothing to its factorisation's backward error
    bp = xp.llt_residual(handle.potrf(A), A) / (m * xp.U)
    for path, b in (('sampler backward', bw), ('potrf of Sigma*+epsI', bp)):
        known = KNOWN.get((path, c.fam, c.n, c.sn))
        record(path, c, b <= 4, known, 'pass' if b <= 4 else 'FAIL', b, b, bl,
               'backward error %.3g m u (bound %s; numpy %.3g m u; jitter %.3g sf2)' % (
                   b, '4' if known is None else '2 x %.3g' % known, bl, eps / c.sf2))
    check_jitter(handle, c, S, eps)
    settle()


@pytest.mark.parametrize('noisy', [False, True])
def test_jitter_rung_on_a_grid_with_duplicates(handle, noisy):
    """S2 where the latent Sigma* is singular: the C5 data of bench_configs (n = 2048, 2-D, l = 20, sf2 = 10,
    sn = 0.25), test points a 30 x 30 grid over the data with 60 of its points repeated."""
    X, y, _ = cfg.make_c5(2048, 1)
    g = np.linspace(0.0, 100.0, 30)
    grid = np.stack(np.meshgrid(g, g, indexing='ij'), axis=-1).reshape(-1, 2)
    Z = np.vstack([grid, grid[::15]])
    kh = np.array([20.0, 20.0, 10.0, 0.0625])
    c = Case(handle, 'C5', 2048, 0.25, len(Z), noisy, X, y, Z, kh, 0)
    _, S = handle.gpr_predict_full(kh, Z, noisy=noisy)
    _, eps = handle.gpr_sample(kh, Z, 4, seed=SEED, noisy=noisy)
    RESULTS.append((noisy or eps > 0, 'no jitter on a latent Sigma* with repeated points'))
    check_jitter(handle, c, S, eps)
    settle()


@pytest.mark.parametrize('nsamp', [1, 129])
@pytest.mark.parametrize('fam,n,sn,m,noisy', CASES, ids=ids(CASES))
def test_samples_are_fz_plus_the_draws(handle, cases, fam, n, sn, m, noisy, nsamp):
    """S3: the mean enters the samples by one add, after the draws."""
    c = cases(fam, n, sn, m, noisy)
    c.train(handle, y=np.zeros(n))
    D, eps0 = handle.gpr_sample(c.khyp, c.Z, nsamp, seed=SEED, kind=c.kind, noisy=noisy)
    c.train(handle)
    fz, _ = handle.gpr_predict_full(c.khyp, c.Z, mean=0.7, kind=c.kind, noisy=noisy)
    s, eps = handle.gpr_sample(c.khyp, c.Z, nsamp, seed=SEED, mean=0.7, kind=c.kind, noisy=noisy)
    assert eps == eps0
    assert np.array_equal(s, fz + D), np.abs(s - (fz + D)).max()
