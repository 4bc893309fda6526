"""Factorisation, solves, prediction and gradient against an extended-precision reference across the conditioning range.

The parity tests compare with the CPU oracle, which assembles its own K; above cond(K) ~ 1e8 one ulp of difference per
entry of K moves the answer by more than their tolerance, so they only run where K is well conditioned.  Users get
much further: optimisers drive log sn down until K is as ill-conditioned as float64 allows.  Here every reference is
computed on the device's OWN matrix (``Handle.kxx`` / ``Handle.kxz``) in long double (tests/_xprec.py), together with
float64 LAPACK on the same matrix, and each device result is held to LAPACK's accuracy:

  C1  |gpu - truth| <= 10 |lapack - truth| + 16 n u scale       (max norms; u = 2^-53; scale: |NLML| for the value,
      max|mean| for the posterior mean, sf2 for the variance, max|g| for the gradient, max|L| for the factor;
      |lapack - truth| is the median over K and 4 symmetric permutations of it, and for L the error on K itself)
  C2  max|L L^T - A| / max|A| <= 4 n u                          (backward error of the factor, in long double)

The device solves triangular systems as products with explicit inverses (32-block and tile inverses, z = W r, K^-1 =
U U^T), which are only conditionally stable.  On the dense 1-D families some checks leave the envelope from cond ~ 1e8
on; they are listed in KNOWN with their measured figure and held to twice it (DESIGN.md 9).  Every check of a test
runs before the test reports, and every message carries the measured gpu/LAPACK ratio.  With
GPB_CONDITIONING_TABLE=<file> the module writes the table of all checks (profiles/r03_conditioning.txt).

Families (n in {128, 200, 384, 512, 1000}: one tile, ragged, several tiles, ragged with 8 tiles):
  F1  squared exponential on dense 1-D inputs, l = 0.3, sf = 1, sn in 1e-1 .. 1e-5   (cond 3e4 .. 3e12; the sweep
      stops at cond ~ 3e12, so n = 1000 (cond 6e12 at sn = 1e-5) ends at sn = 1e-4)
  F2  squared exponential, D = 8, l = 0.5                                            (cond saturates near 1e4: control)
  F3  Matern 3/2, 1-D, sn = 1e-3
  F4  Q diag(lambda) Q^T with a geometric spectrum, cond 1e6 and 1e10               (factorisation only)
"""
import contextlib
import os

import numpy as np
import pytest

from tests import _xprec as xp

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(np.finfo(np.longdouble).eps > 1e-18,
                                 reason='np.longdouble is not wider than float64 here: no extended-precision reference')]

NS = [128, 200, 384, 512, 1000]
GRAD_NS = [128, 200, 384, 512]                 # K^-1 in long double is n^3: the gradient stops at 512
SNS = [1e-1, 1e-2, 1e-3, 1e-4, 1e-5]
F2_SNS = [1e-1, 1e-3, 1e-5]
F2_NS = [128, 512]
OPTION_DEFAULTS = dict(fuse_min_tiles=72, potrf_variant=3, potrf_refine=1)
TABLE = []


# Measured on the B200 (profiles/r03_conditioning.txt): checks outside C1 / C2, keyed (check, family, n, sn), with the
# measured gpu/LAPACK ratio (backward-error checks: the backward error in units of n u).  Such a check is held to twice
# its measured figure instead of the envelope, so a regression there is still caught.  The CPU model of the design's
# order leaves the envelope on the same inputs (tests/test_xprec_reference.py::test_design_model_*, DESIGN.md 9).
KNOWN = {
    ('potrf L default', 'F1', 128, 0.001): 11.4,
    ('potrf backward default', 'F1', 128, 0.0001): 4.98,
    ('potrf backward potrf_refine=0', 'F1', 128, 0.0001): 4.98,
    ('potrf backward default', 'F1', 128, 1e-05): 16.9,
    ('potrf backward potrf_refine=0', 'F1', 128, 1e-05): 17.1,
    ('potrf backward default', 'F1', 200, 0.0001): 11.2,
    ('potrf L default', 'F1', 200, 0.0001): 20,
    ('potrf backward potrf_variant=2', 'F1', 200, 0.0001): 13,
    ('potrf backward potrf_refine=0', 'F1', 200, 0.0001): 10.8,
    ('potrf L potrf_refine=0', 'F1', 200, 0.0001): 38,
    ('potrf backward default', 'F1', 200, 1e-05): 74.9,
    ('potrf L default', 'F1', 200, 1e-05): 97.3,
    ('potrf backward potrf_variant=2', 'F1', 200, 1e-05): 104,
    ('potrf backward potrf_refine=0', 'F1', 200, 1e-05): 63,
    ('potrf L potrf_refine=0', 'F1', 200, 1e-05): 41.5,
    ('potrf L potrf_variant=2', 'F1', 384, 0.001): 11,
    ('potrf L potrf_refine=0', 'F1', 384, 0.001): 12.1,
    ('potrf L default', 'F1', 384, 0.0001): 13.7,
    ('potrf L potrf_variant=2', 'F1', 384, 0.0001): 15.9,
    ('potrf L potrf_refine=0', 'F1', 384, 0.0001): 13.8,
    ('potrf L default', 'F1', 384, 1e-05): 19.8,
    ('potrf L potrf_variant=2', 'F1', 384, 1e-05): 12.7,
    ('potrf L potrf_refine=0', 'F1', 384, 1e-05): 18.2,
    ('potrf backward default', 'F1', 512, 0.0001): 5.31,
    ('potrf L default', 'F1', 512, 0.0001): 15.7,
    ('potrf backward potrf_variant=2', 'F1', 512, 0.0001): 5.99,
    ('potrf L potrf_variant=2', 'F1', 512, 0.0001): 14.9,
    ('potrf backward potrf_refine=0', 'F1', 512, 0.0001): 5.31,
    ('potrf L potrf_refine=0', 'F1', 512, 0.0001): 15.7,
    ('potrf backward default', 'F1', 512, 1e-05): 12.4,
    ('potrf L default', 'F1', 512, 1e-05): 190,
    ('potrf backward potrf_variant=2', 'F1', 512, 1e-05): 11.6,
    ('potrf L potrf_variant=2', 'F1', 512, 1e-05): 168,
    ('potrf backward potrf_refine=0', 'F1', 512, 1e-05): 12.2,
    ('potrf L potrf_refine=0', 'F1', 512, 1e-05): 206,
    ('potrf backward default', 'F1', 1000, 0.0001): 5.7,
    ('potrf L default', 'F3', 1000, 0.001): 13.9,
    ('nlml appended_row', 'F1', 128, 0.0001): 47.3,
    ('nlml fused', 'F1', 128, 0.0001): 47.3,
    ('nlml appended_row', 'F1', 128, 1e-05): 56.1,
    ('nlml fused', 'F1', 128, 1e-05): 56.1,
    ('nlml appended_row', 'F1', 200, 0.001): 16.3,
    ('nlml fused', 'F1', 200, 0.001): 16.3,
    ('nlml appended_row', 'F1', 200, 0.0001): 10.2,
    ('nlml fused', 'F1', 200, 0.0001): 10.2,
    ('nlml appended_row', 'F1', 200, 1e-05): 736,
    ('nlml fused', 'F1', 200, 1e-05): 736,
    ('nlml appended_row', 'F1', 384, 1e-05): 21.7,
    ('nlml fused', 'F1', 384, 1e-05): 21.7,
    ('nlml appended_row', 'F1', 512, 0.001): 11.6,
    ('nlml fused', 'F1', 512, 0.001): 11.6,
    ('nlml appended_row', 'F1', 512, 0.0001): 103,
    ('nlml fused', 'F1', 512, 0.0001): 103,
    ('nlml appended_row', 'F1', 512, 1e-05): 118,
    ('nlml fused', 'F1', 512, 1e-05): 118,
    ('nlml appended_row', 'F1', 1000, 0.0001): 23.5,
    ('nlml fused', 'F1', 1000, 0.0001): 23.5,
    ('predict mean', 'F1', 128, 0.0001): 22,
    ('predict mean', 'F1', 128, 1e-05): 139,
    ('predict mean', 'F1', 200, 0.0001): 23.1,
    ('predict mean', 'F1', 200, 1e-05): 449,
    ('predict mean', 'F1', 512, 0.001): 11.3,
    ('predict mean', 'F1', 512, 0.0001): 76.9,
    ('predict mean', 'F1', 512, 1e-05): 127,
    ('predict mean', 'F1', 1000, 0.0001): 26,
    ('grad value', 'F1', 128, 0.0001): 47.3,
    ('grad gradient', 'F1', 128, 0.0001): 35.2,
    ('grad value', 'F1', 128, 1e-05): 56.1,
    ('grad gradient', 'F1', 128, 1e-05): 56.2,
    ('grad value', 'F1', 200, 0.001): 16.3,
    ('grad value', 'F1', 200, 0.0001): 10.2,
    ('grad gradient', 'F1', 200, 0.0001): 10.4,
    ('grad value', 'F1', 200, 1e-05): 736,
    ('grad gradient', 'F1', 200, 1e-05): 697,
    ('grad value', 'F1', 384, 1e-05): 21.7,
    ('grad gradient', 'F1', 384, 1e-05): 21.3,
    ('grad value', 'F1', 512, 0.001): 11.6,
    ('grad gradient', 'F1', 512, 0.001): 11.7,
    ('grad value', 'F1', 512, 0.0001): 103,
    ('grad gradient', 'F1', 512, 0.0001): 104,
    ('grad value', 'F1', 512, 1e-05): 118,
    ('grad gradient', 'F1', 512, 1e-05): 131,
    ('batched value', 'F1', 384, 1e-05): 21.7,
    ('batched+grad value', 'F1', 384, 1e-05): 21.7,
    ('batched gradient', 'F1', 384, 1e-05): 21.3,
    ('batched B=70 value', 'F1#3', 200, 0.0001): 10.2,
    ('batched B=70 gradient', 'F1#3', 200, 0.0001): 10.4,
    ('batched B=70 value', 'F1#4', 200, 0.001): 13.8,
    ('grow value', 'F1', 150, 0.001): 16.4,
    ('grow value', 'F1', 333, 0.001): 29.9,
    ('grow value', 'F1', 512, 0.001): 12,
    ('grow predict mean', 'F1', 512, 0.001): 11.3,
    ('grow value', 'F1', 150, 0.0001): 19.2,
    ('grow value', 'F1', 333, 0.0001): 123,
    ('grow value', 'F1', 512, 0.0001): 102,
    ('grow predict mean', 'F1', 512, 0.0001): 76.9,
}
RESULTS = []


@pytest.fixture(autouse=True)
def _results():
    RESULTS.clear()
    yield


@contextlib.contextmanager
def options(handle, **kv):
    try:
        for k, v in kv.items():
            handle.set_option(k, v)
        yield
    finally:
        for k in kv:
            handle.set_option(k, OPTION_DEFAULTS[k])


inputs = xp.gp_inputs


def spectrum_matrix(n, cond, seed=0):
    """F4: Q diag(lambda) Q^T, lambda geometric from 1 to 1/cond."""
    rng = np.random.default_rng(seed + n)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    A = (Q * np.geomspace(1.0, 1.0 / cond, n)) @ Q.T
    return (A + A.T) / 2


class Case:
    """One matrix with both solvers of it; the long-double work is done once, on first use."""

    def __init__(self, fam, n, sn, K, X=None, y=None, Z=None, khyp=None, kind=0, Kxz=None):
        self.fam, self.n, self.sn, self.K = fam, n, sn, K
        self.X, self.y, self.Z, self.khyp, self.kind, self.Kxz = X, y, Z, khyp, kind, Kxz
        ev = np.linalg.eigvalsh(K)
        self.cond = ev[-1] / ev[0] if ev[0] > 0 else np.inf
        self._memo = {}

    def memo(self, key, f):
        if key not in self._memo:
            self._memo[key] = f()
        return self._memo[key]

    @property
    def exact(self):
        return self.memo('E', lambda: xp.Exact(self.K))

    @property
    def lapack(self):
        return self.memo('P', lambda: xp.Lapack(self.K))

    def samples(self, key, f):
        """LAPACK's value of a quantity on K and on 4 symmetric permutations of it (xp.lapack_samples)."""
        return self.memo('s_' + key, lambda: xp.lapack_samples(self.K, f))

    def nlml(self):
        return self.memo('nlml', lambda: (self.exact.nlml(self.y),
                                          self.samples('nlml', lambda P, p: P.nlml(self.y[p]))))

    def predict(self):
        sf2 = self.khyp[-2]
        truth = self.memo('pred', lambda: self.exact.predict(self.y, self.Kxz, sf2))
        lap = self.samples('pred', lambda P, p: P.predict(self.y[p], self.Kxz[p], sf2))
        return truth, ([m for m, _ in lap], [v for _, v in lap])

    def grad(self):
        return self.memo('grad', lambda: (self.exact.se_grad(self.X, self.y, self.khyp),
                                          self.samples('grad', lambda P, p: P.se_grad(self.X[p], self.y[p], self.khyp))))

    def train(self, handle):
        handle.set_train(self.X, self.y)

    def label(self):
        return '%s n=%d %s' % (self.fam, self.n, 'cond=%.0e' % self.sn if self.fam == 'F4' else 'sn=%.0e' % self.sn)


def check(path, case, got, lapack, truth, scale):
    """C1 (or, for a KNOWN case, twice its measured ratio), recorded in the table and in RESULTS; ``settle`` asserts."""
    ok, ratio, eg, el = xp.forward_check(got, lapack, truth, case.n, scale)
    known = KNOWN.get((path, case.fam, case.n, case.sn))
    status = 'pass' if ok else 'FAIL'
    if known is not None:
        status = 'known %.3g' % known
        ok = ratio <= 2 * known
    TABLE.append((path, case, ratio, eg, el, status if ok else 'FAIL (' + status + ')'))
    RESULTS.append((ok, '%s, %s (cond %.1e): gpu/LAPACK error ratio %.3g (gpu %.3g, LAPACK %.3g, floor %.3g)%s' % (
        path, case.label(), case.cond, ratio, eg, el, 16 * case.n * xp.U * scale,
        '' if known is None else ', measured before %.3g' % known)))
    return ratio


def check_backward(path, case, L):
    """C2 (or, for a KNOWN case, twice its measured figure) on the factor; LAPACK's own backward error in the table."""
    n = case.n
    bw = xp.llt_residual(L, case.K) / (n * xp.U)
    bl = case.memo('bw_lapack', lambda: xp.llt_residual(case.lapack.L, case.K) / (n * xp.U))
    known = KNOWN.get((path, case.fam, n, case.sn))
    ok = bw <= 4 if known is None else bw <= 2 * known
    status = ('pass' if bw <= 4 else 'FAIL') if known is None else 'known %.3g' % known
    TABLE.append((path, case, bw, bw, bl, status if ok else 'FAIL (' + status + ')'))
    RESULTS.append((ok, '%s, %s (cond %.1e): backward error %.3g n u (bound %s; LAPACK %.3g n u)' % (
        path, case.label(), case.cond, bw, '4' if known is None else '2 x %.3g' % known, bl)))


def settle():
    """Every check of the test has run: report all that failed."""
    bad = [m for ok, m in RESULTS if not ok]
    assert not bad, '\n'.join(bad)


@pytest.fixture(scope='module')
def cases(handle):
    """case(fam, n, sn): the device's K (and Kxz) of that problem and the references on them, built once per module."""
    cache = {}

    def get(fam, n, sn):
        key = (fam, n, sn)
        if key not in cache:
            if fam == 'F4':
                cache[key] = Case(fam, n, sn, spectrum_matrix(n, sn))
            else:
                X, y, Z, kh, kind = inputs(fam, n, sn)
                handle.set_train(X, y)
                cache[key] = Case(fam, n, sn, handle.kxx(kh, kind=kind), X, y, Z, kh, kind, handle.kxz(kh, Z, kind=kind))
        return cache[key]

    yield get
    path = os.environ.get('GPB_CONDITIONING_TABLE')
    if path:
        write_table(path)


def write_table(path):
    import torch
    lines = ['# tests/test_gpu_conditioning.py on %s: device error / float64 LAPACK error, both against the long-double'
             % torch.cuda.get_device_name(0),
             '# reference on the device\'s own matrix (C1 passes at ratio <= 10 or under the floor 16 n u scale).',
             '# LAPACK error: median over K and 4 symmetric permutations of it.  "known r": outside the envelope, held to 2 r.',
             '# backward rows: max|LL^T - A|/max|A| in units of n u for the device and for LAPACK (C2: device <= 4).',
             '%-30s %-6s %5s %-10s %9s %10s %10s %9s %s' % ('check', 'fam', 'n', 'sn/cond', 'cond(K)', 'err gpu',
                                                            'err lapack', 'ratio', 'status')]
    for path_, c, ratio, eg, el, status in TABLE:
        lines.append('%-30s %-6s %5d %-10.0e %9.1e %10.3g %10.3g %9.3g %s' % (
            path_, c.fam, c.n, c.sn, c.cond, eg, el, ratio, status))
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, 'w') as f:
        f.write('\n'.join(lines) + '\n')


def gp_params(families=('F1', 'F2', 'F3'), ns=NS, f1_sns=SNS):
    out = []
    for fam in families:
        if fam == 'F1':
            out += [(fam, n, sn) for n in ns for sn in f1_sns if not (n > 512 and sn < 1e-4)]
        elif fam == 'F2':
            out += [(fam, n, sn) for n in ns if n in F2_NS for sn in F2_SNS]
        elif fam == 'F3':
            out += [(fam, n, 1e-3) for n in ns]
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the matrices themselves
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('fam,n,sn', [('F1', 200, 1e-3), ('F2', 128, 1e-3), ('F3', 200, 1e-3)])
def test_kxx_off_diagonal_is_kxz_of_the_training_points(handle, fam, n, sn):
    """The assembly kernel (se_ard.cu) runs the same element code in its symmetric and rectangular modes, so K of the
    fits and Kxz of the predictions are the same function of the inputs: bit for bit, off the diagonal and, with the
    noise added once, on it.  The references below rely on this."""
    X, y, _, kh, kind = inputs(fam, n, sn)
    handle.set_train(X, y)
    K = handle.kxx(kh, kind=kind)
    Kz = handle.kxz(kh, X, kind=kind)
    off = ~np.eye(n, dtype=bool)
    assert np.array_equal(K[off], Kz[off])
    assert np.array_equal(np.diagonal(K), np.diagonal(Kz) + kh[-1])


# ---------------------------------------------------------------------------------------------------------------------
# factorisation
# ---------------------------------------------------------------------------------------------------------------------
POTRF_VARIANTS = {'default': {}, 'potrf_variant=2': dict(potrf_variant=2), 'potrf_refine=0': dict(potrf_refine=0)}


def potrf_params():
    out = []
    for fam, n, sn in gp_params() + [('F4', n, c) for n in NS for c in (1e6, 1e10)]:
        for v in POTRF_VARIANTS:
            if v == 'default' or n <= 512:
                out.append((fam, n, sn, v))
    return out


@pytest.mark.parametrize('fam,n,sn,variant', potrf_params())
def test_potrf_backward_and_forward_error(handle, cases, fam, n, sn, variant):
    c = cases(fam, n, sn)
    with options(handle, **POTRF_VARIANTS[variant]):
        L = handle.potrf(c.K)
    check_backward('potrf backward ' + variant, c, L)
    check('potrf L ' + variant, c, L, c.lapack.L, c.exact.L, float(np.abs(c.exact.L).max()))
    settle()


@pytest.mark.parametrize('n', [128, 200, 512])
@pytest.mark.parametrize('cond', [1e6, 1e10])
def test_potrf_commutes_with_power_of_4_scaling(handle, n, cond):
    """Every step of the factorisation is exact under A -> 4^k A (L -> 2^k L) unless the pivot's rsqrt.approx.ftz
    or the updates misbehave near the ends of the exponent range: 2 ulp per entry at most (bit for bit expected)."""
    A = spectrum_matrix(n, cond)
    L = handle.potrf(A)
    for k in (60, -60, 240, -240):
        Lc = handle.potrf(np.ldexp(A, 2 * k))
        ref = np.ldexp(L, k)
        ulps = np.abs(Lc - ref) / np.spacing(np.abs(ref))
        assert np.isfinite(Lc).all() and ulps.max() <= 2, (k, ulps.max(), np.count_nonzero(ulps))


@pytest.mark.parametrize('n', [128, 384, 512])
def test_potrf_dev_with_padded_leading_dimension(handle, cases, n):
    """gpb_potrf_lower_dev with lda = n + 64: the columns past n are never touched, and the factor is bit for bit the
    lda = n one (which is also what the host entry point returns)."""
    import torch
    c = cases('F1', n, 1e-3)
    Kt = torch.from_numpy(c.K).cuda()
    W = Kt.clone()
    P = torch.full((n, n + 64), float('nan'), dtype=torch.float64, device='cuda')
    P[:, :n] = Kt
    torch.cuda.synchronize()
    assert handle.potrf_dev(W.data_ptr(), n, n) == 0
    assert handle.potrf_dev(P.data_ptr(), n, n + 64) == 0
    torch.cuda.synchronize()
    assert torch.isnan(P[:, n:]).all()
    L1, L2 = torch.tril(W).cpu().numpy(), torch.tril(P[:, :n]).cpu().numpy()
    assert np.array_equal(L1, L2)
    assert np.array_equal(L1, handle.potrf(c.K))


# ---------------------------------------------------------------------------------------------------------------------
# value, prediction, gradient
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('path', ['appended_row', 'fused'])
@pytest.mark.parametrize('fam,n,sn', gp_params())
def test_nlml(handle, cases, fam, n, sn, path):
    """gpr_nlml: the right-hand side as a row appended under K (the default below 72 tiles) or riding on the
    factorisation (diagonal-tile kernel + panel TRSM epilogue, forced here with fuse_min_tiles = 1)."""
    c = cases(fam, n, sn)
    c.train(handle)
    with options(handle, **(dict(fuse_min_tiles=1) if path == 'fused' else {})):
        v = handle.gpr_nlml(c.khyp, kind=c.kind)
    truth, lap = c.nlml()
    check('nlml ' + path, c, v, lap, truth, abs(float(truth)))
    settle()


@pytest.mark.parametrize('fam,n,sn', gp_params())
def test_predict(handle, cases, fam, n, sn):
    c = cases(fam, n, sn)
    c.train(handle)
    fz, var = handle.gpr_predict(c.khyp, c.Z, kind=c.kind)
    (mt, vt), (ml, vl) = c.predict()
    check('predict mean', c, fz, ml, mt, float(np.abs(mt).max()))
    check('predict variance', c, var, vl, vt, c.khyp[-2])
    settle()


@pytest.mark.parametrize('fam,n,sn', gp_params(('F1', 'F2'), ns=GRAD_NS))
def test_gradient(handle, cases, fam, n, sn):
    """gpr_nlml(want_grad=True): K^-1 = U U^T with U = L^-T swept from an identity block (grad.cu)."""
    c = cases(fam, n, sn)
    c.train(handle)
    v, g = handle.gpr_nlml(c.khyp, want_grad=True)
    truth, lap = c.nlml()
    gt, gl = c.grad()
    check('grad value', c, v, lap, truth, abs(float(truth)))
    check('grad gradient', c, g, gl, gt, float(np.abs(gt).max()))
    settle()


def test_batched_mixed_conditioning(handle, cases):
    """All of F1's noise levels (cond 3e4 .. 3e12) in one batched call, with and without gradients."""
    n = 384
    cs = [cases('F1', n, sn) for sn in SNS]
    cs[0].train(handle)
    kh = np.array([c.khyp for c in cs])
    vals, info = handle.gpr_nlml_batched(kh)
    gvals, grads, ginfo = handle.gpr_nlml_batched(kh, want_grad=True)
    assert not info.any() and not ginfo.any()
    for b, c in enumerate(cs):
        truth, lap = c.nlml()
        gt, gl = c.grad()
        check('batched value', c, vals[b], lap, truth, abs(float(truth)))
        check('batched+grad value', c, gvals[b], lap, truth, abs(float(truth)))
        check('batched gradient', c, grads[b], gl, gt, float(np.abs(gt).max()))
    settle()


def test_batched_member_that_is_not_positive_definite(handle):
    """A member without noise on duplicated inputs fails its factorisation (info > 0); the other members are bit for
    bit what the same call gives with that member replaced by a positive definite one (same size, same schedule)."""
    X, y, _, kh, _ = inputs('F1', 200, 1e-3)
    X[-12:] = X[:12]                                    # duplicated inputs
    handle.set_train(X, y)
    sns = [1e-1, 1e-2, 1e-3, 0.0, 1e-4]
    bad = np.array([np.r_[kh[:2], s * s] for s in sns])
    good = bad.copy()
    good[3, -1] = 1e-4
    for grad in (False, True):
        rb = handle.gpr_nlml_batched(bad, want_grad=grad)
        rg = handle.gpr_nlml_batched(good, want_grad=grad)
        ib, ig = rb[-1], rg[-1]
        assert ib[3] > 0 and not np.delete(ib, 3).any() and not ig.any(), (ib, ig)
        for a, b in zip(rb[:-1], rg[:-1]):
            assert np.array_equal(np.delete(a, 3, axis=0), np.delete(b, 3, axis=0)), grad


def test_batched_gradients_across_the_chunk_boundary(handle):
    """B = 70 > the 64 problems the gradient path keeps resident at once, five distinct hyper-parameter vectors
    cycled so that neighbouring rows differ: every row against the reference of its own matrix, and the rows on
    either side of the boundary that share hyper-parameters (b and b + 5, b = 59..63) bit for bit equal."""
    n = 200
    X, y, _, _, _ = inputs('F1', n, 1e-3)
    handle.set_train(X, y)
    hyps = [(0.3, 1.0, 1e-1), (0.25, 1.3, 1e-2), (0.35, 0.8, 1e-3), (0.3, 1.0, 1e-4), (0.45, 1.1, 1e-3)]
    khs = [np.array([l, sf * sf, sn * sn]) for l, sf, sn in hyps]
    refs = []
    for (l, sf, sn), kh in zip(hyps, khs):
        c = Case('F1#%d' % len(refs), n, sn, handle.kxx(kh), X, y, None, kh)
        refs.append((c, c.nlml(), c.grad()))
    B = 70
    vals, grads, info = handle.gpr_nlml_batched(np.array([khs[b % 5] for b in range(B)]), want_grad=True)
    assert not info.any()
    for b in range(B):
        c, (truth, lap), (gt, gl) = refs[b % 5]
        check('batched B=70 value', c, vals[b], lap, truth, abs(float(truth)))
        check('batched B=70 gradient', c, grads[b], gl, gt, float(np.abs(gt).max()))
    for b in range(59, 64):
        same = vals[b] == vals[b + 5] and np.array_equal(grads[b], grads[b + 5])
        RESULTS.append((same, 'rows %d and %d (same hyper-parameters, chunks 0 and 1) differ: %r %r / %r %r' % (
            b, b + 5, vals[b], vals[b + 5], grads[b], grads[b + 5])))
    settle()


@pytest.mark.parametrize('sn', [1e-3, 1e-4])
def test_growing_set(handle, cases, sn):
    """grow_begin / grow_append in three pieces (the stored factor extended twice), then grow_predict."""
    c = cases('F1', 512, sn)
    handle.grow_begin(c.khyp, 1, capacity=512)
    for a, b in ((0, 150), (150, 333), (333, 512)):
        v = handle.grow_append(c.X[a:b], c.y[a:b])
        sub = c if b == 512 else Case('F1', b, sn, c.K[:b, :b], c.X[:b], c.y[:b], None, c.khyp)
        truth, lap = sub.nlml()
        check('grow value', sub, v, lap, truth, abs(float(truth)))
    fz, var = handle.grow_predict(c.Z)
    (mt, vt), (ml, vl) = c.predict()
    check('grow predict mean', c, fz, ml, mt, float(np.abs(mt).max()))
    check('grow predict variance', c, var, vl, vt, c.khyp[-2])
    settle()


def test_criterion_detects_a_100_ulp_perturbation(handle, cases):
    """The criteria have teeth: on a case the device passes (F1, n = 384, sn = 1e-4, cond 2e10), take the reference
    and LAPACK of K + dK instead, dK a random symmetric perturbation of 100 ulp per entry, while the device still
    factors K.  C1 must then fail, by far: the criterion sees a kernel defect that acts like a backward error of
    100 u, far below what the oracle parity tests resolve at this conditioning.  Three seeded perturbations, each
    must be caught."""
    c = cases('F1', 384, 1e-4)
    c.train(handle)
    v = handle.gpr_nlml(c.khyp)
    truth, lap = c.nlml()
    check('nlml (control, K)', c, v, lap, truth, abs(float(truth)))
    ratios = []
    for seed in range(3):
        S = np.sign(np.random.default_rng(seed).standard_normal(c.K.shape))
        S = np.triu(S) + np.triu(S, 1).T
        p = Case('F1', 384, 1e-4, c.K + 100 * np.spacing(np.abs(c.K)) * S, c.X, c.y, c.Z, c.khyp)
        truth, lap = p.nlml()
        ok, ratio, eg, el = xp.forward_check(v, lap, truth, p.n, abs(float(truth)))
        TABLE.append(('nlml vs K+100ulp #%d' % seed, p, ratio, eg, el, 'caught' if not ok else 'MISSED'))
        ratios.append(ratio)
    RESULTS.append((min(ratios) > 10, 'a 100-ulp backward error went unnoticed: gpu/LAPACK ratios %s' % ratios))
    settle()
