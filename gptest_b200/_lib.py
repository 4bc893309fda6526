"""ctypes binding of libgpb200.so (the C ABI declared in include/gpb200.h).

There is no CPU fallback: if the shared library is missing it is an ImportError-like
RuntimeError telling how to build it, and if no B200 is present ``Handle()`` raises with the
library's own message.
"""
import ctypes as C
import os
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('GPB200_LIB') or os.path.join(_HERE, 'libgpb200.so')     # GPB200_LIB: A/B of two builds (tools/)
CSRC = os.path.join(_HERE, 'csrc')

_lib = None
_lock = threading.Lock()

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int32)
c_lp = C.POINTER(C.c_int64)
c_fp = C.POINTER(C.c_float)

# name -> (restype, argtypes): exactly the declarations of include/gpb200.h
SIGNATURES = {
    'gpb_version': (C.c_int, []),
    'gpb_create': (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    'gpb_set_stream': (C.c_int, [C.c_void_p, C.c_void_p]),
    'gpb_get_stream': (C.c_void_p, [C.c_void_p]),
    'gpb_destroy': (C.c_int, [C.c_void_p]),
    'gpb_last_error': (C.c_char_p, [C.c_void_p]),
    'gpb_set_option': (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    'gpb_get_timings': (C.c_int, [C.c_void_p, c_fp, C.c_int]),
    'gpb_launch_count': (C.c_int64, [C.c_void_p]),
    'gpb_set_train': (C.c_int, [C.c_void_p, c_dp, C.c_int64, C.c_int32, c_dp]),
    'gpb_set_train_dev': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    'gpb_se_ard_kxx': (C.c_int, [C.c_void_p, c_dp, C.c_void_p, C.c_int32, C.c_int32]),
    'gpb_se_ard_kxz': (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int64, C.c_void_p, C.c_int32]),
    'gpb_sqdist': (C.c_int, [C.c_void_p, c_dp, C.c_int64, c_dp]),
    'gpb_gpr_nlml': (C.c_int, [C.c_void_p, c_dp, C.c_double, c_dp, c_dp, c_ip]),
    'gpb_gpr_predict': (C.c_int, [C.c_void_p, c_dp, C.c_double, c_dp, C.c_int64, c_dp, c_dp, c_ip]),
    'gpb_gpr_predict_full': (C.c_int, [C.c_void_p, c_dp, C.c_double, c_dp, C.c_int64, c_dp, C.c_void_p, C.c_int32,
                                       C.c_int32, c_ip]),
    'gpb_gpr_sample': (C.c_int, [C.c_void_p, c_dp, C.c_double, c_dp, C.c_int64, C.c_int64, C.c_uint64, C.c_int32,
                                 c_dp, c_dp, c_ip]),
    'gpb_gpr_nlml_batched': (C.c_int, [C.c_void_p, c_dp, C.c_int64, C.c_double, c_dp, c_dp, c_ip]),
    'gpb_gpr_grow_begin': (C.c_int, [C.c_void_p, c_dp, C.c_int32, C.c_double, C.c_int64]),
    'gpb_gpr_grow_append': (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int64, c_dp, c_ip]),
    'gpb_gpr_grow_predict': (C.c_int, [C.c_void_p, c_dp, C.c_int64, c_dp, c_dp]),
    'gpb_gpr_grow_size': (C.c_int64, [C.c_void_p]),
    'gpb_potrf_lower_dev': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, c_ip]),
    'gpb_potrf_lower': (C.c_int, [C.c_void_p, c_dp, C.c_int64, c_ip]),
    'gpb_dgemm_nt_dev': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                   C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_double]),
    'gpb_gpc_laplace': (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int32, C.c_double, C.c_int32, C.c_int32, c_dp,
                                  c_dp, c_ip, c_dp, c_dp, c_ip]),
    'gpb_gpc_predict': (C.c_int, [C.c_void_p, c_dp, C.c_int64, c_dp, c_dp, c_dp]),
    'gpb_gpc_evidence_grad': (C.c_int, [C.c_void_p, c_dp, c_dp]),
    'gpb_pref_laplace': (C.c_int, [C.c_void_p, c_lp, c_dp, C.c_int64, c_dp, C.c_double, C.c_double, C.c_int32,
                                   C.c_int32, C.c_int32, c_dp, c_dp, c_ip, c_dp, c_dp, c_ip]),
    'gpb_pref_log_marginal': (C.c_int, [C.c_void_p, c_lp, c_dp, C.c_int64, C.c_int64, c_dp, c_dp, C.c_double, C.c_double, c_dp]),
    'gpb_pref_evidence': (C.c_int, [C.c_void_p, c_dp]),
    'gpb_pref_evidence_grad': (C.c_int, [C.c_void_p, c_dp, c_dp]),
    'gpb_pref_predict': (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int64, c_dp, c_dp, c_dp]),
    'gpb_pref_derivatives': (C.c_int, [C.c_void_p, c_lp, c_dp, C.c_int64, C.c_int64, c_dp, C.c_double,
                                       C.c_int32, c_dp, c_dp]),
    'gpb_microbench': (C.c_int, [C.c_void_p, C.c_int32, c_dp]),
}


def build(verbose=False):
    """Compile libgpb200.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(['make', '-j8', '-C', CSRC], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode:
        raise RuntimeError('building libgpb200.so failed')
    return LIB_PATH


def load():
    """Load the shared library (once) and attach the prototypes."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                'libgpb200.so is not built (%s). Run `python -c "import __graft_entry__ as g; g.build()"` '
                'or `make -C gptest_b200/csrc`. There is no CPU fallback.' % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


class GpbError(RuntimeError):
    pass


def _dp(a):
    return a.ctypes.data_as(c_dp)


def as_f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


class Handle:
    """One device + one stream + resident work space (a gpb_handle)."""

    def __init__(self, device=0):
        self.lib = load()
        hp = C.c_void_p()
        rc = self.lib.gpb_create(int(device), C.byref(hp))
        if rc != 0:
            raise GpbError('gpb_create failed: %s' % self.lib.gpb_last_error(None).decode())
        self.h = hp
        self.device = device
        self._cov_kind = 0

    def close(self):
        if getattr(self, 'h', None):
            self.lib.gpb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != 0:
            raise GpbError('libgpb200 error %d: %s' % (rc, self.lib.gpb_last_error(self.h).decode()))

    # ---- plumbing --------------------------------------------------------------------------
    def set_stream(self, stream_ptr):
        self.check(self.lib.gpb_set_stream(self.h, C.c_void_p(stream_ptr)))

    def stream(self):
        return self.lib.gpb_get_stream(self.h) or 0

    def set_option(self, name, value):
        self.check(self.lib.gpb_set_option(self.h, name.encode(), int(value)))

    def timings(self):
        buf = (C.c_float * 8)()
        self.lib.gpb_get_timings(self.h, buf, 8)
        t = list(buf)
        return dict(kbuild_ms=t[0], factor_ms=t[1], finish_ms=t[2], grad_ms=t[3], total_ms=t[4])

    def launch_count(self):
        return int(self.lib.gpb_launch_count(self.h))

    # ---- data ------------------------------------------------------------------------------
    def set_train(self, X, y=None):
        X = as_f64(X)
        X = X.reshape(len(X), -1)
        yp = None
        if y is not None:
            y = as_f64(y).reshape(-1)
            assert len(y) == len(X)
            yp = _dp(y)
        self.n, self.d = X.shape
        self.check(self.lib.gpb_set_train(self.h, _dp(X), X.shape[0], X.shape[1], yp))

    # ---- covariance --------------------------------------------------------------------------
    # ``kind``: 0 squared exponential (the reference's only kernel, GPr.py:90-110), 1 Matern 3/2, 2 Matern 5/2.
    # It is a handle option on the C side; every wrapper sets it, so the default is always the reference's kernel.
    def _khyp(self, khyp, extra=2):
        """khyp as fp64 with d + extra entries per row; the C side reads khyp[.. d + extra - 1] unconditionally, so a
        vector that does not fit the input dimension is refused here (the reference fails with a numpy
        broadcasting ValueError in the same situation)."""
        khyp = as_f64(khyp)
        if not hasattr(self, 'd'):
            raise ValueError('no training data on this handle: call set_train first')
        if khyp.shape[-1] != self.d + extra:
            raise ValueError('hyper-parameter vector has %d entries, input dimension %d needs %d'
                             % (khyp.shape[-1], self.d, self.d + extra))
        return khyp

    def _kind(self, kind):
        if kind != self._cov_kind:
            self.check(self.lib.gpb_set_option(self.h, b'cov_kind', int(kind)))
            self._cov_kind = kind

    def kxx(self, khyp, flags=0, kind=0):
        self._kind(kind)
        khyp = self._khyp(khyp)
        out = np.empty((self.n, self.n))
        self.check(self.lib.gpb_se_ard_kxx(self.h, _dp(khyp), out.ctypes.data_as(C.c_void_p), 0, flags))
        return out

    def kxx_dev(self, khyp, dev_ptr, flags=0, kind=0):
        self._kind(kind)
        khyp = self._khyp(khyp)
        self.check(self.lib.gpb_se_ard_kxx(self.h, _dp(khyp), C.c_void_p(dev_ptr), 1, flags))

    def kxz(self, khyp, Z, kind=0):
        self._kind(kind)
        khyp = self._khyp(khyp)
        Z = as_f64(Z)
        Z = Z.reshape(len(Z), -1)
        out = np.empty((self.n, Z.shape[0]))
        self.check(self.lib.gpb_se_ard_kxz(self.h, _dp(khyp), _dp(Z), Z.shape[0], out.ctypes.data_as(C.c_void_p), 0))
        return out

    def sqdist(self, B):
        B = as_f64(B)
        B = B.reshape(len(B), -1)
        out = np.empty((self.n, B.shape[0]))
        self.check(self.lib.gpb_sqdist(self.h, _dp(B), B.shape[0], _dp(out)))
        return out

    # ---- regression ----------------------------------------------------------------------------
    def gpr_nlml(self, khyp, mean=0.0, want_grad=False, kind=0):
        self._kind(kind)
        khyp = self._khyp(khyp)
        val = C.c_double()
        info = C.c_int32()
        grad = np.empty(len(khyp)) if want_grad else None
        self.check(self.lib.gpb_gpr_nlml(self.h, _dp(khyp), float(mean), C.byref(val),
                                         _dp(grad) if want_grad else None, C.byref(info)))
        if info.value > 0:
            raise np.linalg.LinAlgError('Matrix is not positive definite (leading minor %d)' % info.value)
        return (val.value, grad) if want_grad else val.value

    def gpr_predict(self, khyp, Z, mean=0.0, kind=0):
        self._kind(kind)
        khyp = self._khyp(khyp)
        Z = as_f64(Z)
        Z = Z.reshape(len(Z), -1)
        m = Z.shape[0]
        fz, cov = np.empty(m), np.empty(m)
        info = C.c_int32()
        self.check(self.lib.gpb_gpr_predict(self.h, _dp(khyp), float(mean), _dp(Z), m, _dp(fz), _dp(cov), C.byref(info)))
        if info.value > 0:
            raise np.linalg.LinAlgError('Matrix is not positive definite (leading minor %d)' % info.value)
        return fz, cov

    def gpr_predict_full(self, khyp, Z, mean=0.0, kind=0, noisy=False):
        """(fz (m,), cov (m, m)): fz as gpr_predict, cov the joint posterior covariance of the latent f at Z, plus
        sn2 I with noisy=True (the predictive of noisy observations)."""
        self._kind(kind)
        khyp = self._khyp(khyp)
        Z = as_f64(Z)
        Z = Z.reshape(len(Z), -1)
        m = Z.shape[0]
        fz, cov = np.empty(m), np.empty((m, m))
        info = C.c_int32()
        self.check(self.lib.gpb_gpr_predict_full(self.h, _dp(khyp), float(mean), _dp(Z), m, _dp(fz),
                                                 cov.ctypes.data_as(C.c_void_p), 0, 1 if noisy else 0, C.byref(info)))
        if info.value > 0:
            raise np.linalg.LinAlgError('Matrix is not positive definite (leading minor %d)' % info.value)
        return fz, cov

    def gpr_sample(self, khyp, Z, nsamp, seed=0, mean=0.0, kind=0, noisy=False):
        """(samples (nsamp, m), jitter): joint draws fz + L e with L L^T = cov + jitter I (cov of gpr_predict_full);
        the normals e are a function of (seed, sample, point) alone."""
        self._kind(kind)
        khyp = self._khyp(khyp)
        Z = as_f64(Z)
        Z = Z.reshape(len(Z), -1)
        m = Z.shape[0]
        out = np.empty((int(nsamp), m))
        jit = C.c_double()
        info = C.c_int32()
        self.check(self.lib.gpb_gpr_sample(self.h, _dp(khyp), float(mean), _dp(Z), m, int(nsamp),
                                           int(seed) & 0xFFFFFFFFFFFFFFFF, 1 if noisy else 0, _dp(out), C.byref(jit),
                                           C.byref(info)))
        if info.value > 0:
            raise np.linalg.LinAlgError('Matrix is not positive definite (leading minor %d)' % info.value)
        return out, jit.value

    def gpr_nlml_batched(self, khyp, mean=0.0, want_grad=False, kind=0):
        self._kind(kind)
        khyp = self._khyp(np.atleast_2d(as_f64(khyp)))
        B, p = khyp.shape
        val = np.empty(B)
        info = np.zeros(B, dtype=np.int32)
        grad = np.empty((B, p)) if want_grad else None
        self.check(self.lib.gpb_gpr_nlml_batched(self.h, _dp(khyp), B, float(mean), _dp(val),
                                                 _dp(grad) if want_grad else None, info.ctypes.data_as(c_ip)))
        return (val, grad, info) if want_grad else (val, info)

    # ---- growing training set (GP_parameter_fit.py:61-63) --------------------------------------
    def grow_begin(self, khyp, d, capacity, mean=0.0, kind=0):
        self._kind(kind)
        khyp = as_f64(khyp).reshape(-1)
        assert khyp.size == d + 2
        self.check(self.lib.gpb_gpr_grow_begin(self.h, _dp(khyp), int(d), float(mean), int(capacity)))

    def grow_append(self, X_new, y_new):
        X_new = as_f64(X_new)
        X_new = X_new.reshape(len(X_new), -1)
        y_new = as_f64(y_new).reshape(-1)
        assert len(X_new) == len(y_new)
        val = np.empty(1)
        info = C.c_int32()
        self.check(self.lib.gpb_gpr_grow_append(self.h, _dp(X_new), _dp(y_new), len(y_new), _dp(val), C.byref(info)))
        if info.value > 0:
            raise np.linalg.LinAlgError('Matrix is not positive definite (leading minor %d)' % info.value)
        return float(val[0])

    def grow_predict(self, Z):
        Z = as_f64(Z)
        Z = Z.reshape(len(Z), -1)
        fz = np.empty(len(Z))
        cov = np.empty(len(Z))
        self.check(self.lib.gpb_gpr_grow_predict(self.h, _dp(Z), len(Z), _dp(fz), _dp(cov)))
        return fz, cov

    def grow_size(self):
        return int(self.lib.gpb_gpr_grow_size(self.h))

    # ---- dense hooks ------------------------------------------------------------------------
    def potrf(self, A):
        A = np.array(A, dtype=np.float64, order='C')
        info = C.c_int32()
        self.check(self.lib.gpb_potrf_lower(self.h, _dp(A), A.shape[0], C.byref(info)))
        if info.value > 0:
            raise np.linalg.LinAlgError('Matrix is not positive definite (leading minor %d)' % info.value)
        return A

    def potrf_dev(self, dev_ptr, n, lda):
        info = C.c_int32()
        self.check(self.lib.gpb_potrf_lower_dev(self.h, C.c_void_p(dev_ptr), n, lda, C.byref(info)))
        return info.value

    def dgemm_nt_dev(self, c_ptr, ldc, a_ptr, lda, b_ptr, ldb, M, N, K, alpha, beta):
        self.check(self.lib.gpb_dgemm_nt_dev(self.h, C.c_void_p(c_ptr), ldc, C.c_void_p(a_ptr), lda,
                                             C.c_void_p(b_ptr), ldb, M, N, K, alpha, beta))

    def microbench(self, kind):
        v = C.c_double()
        self.check(self.lib.gpb_microbench(self.h, kind, C.byref(v)))
        return v.value


_default = {}
_default_device = int(os.environ.get('GPB_DEVICE', os.environ.get('LOCAL_RANK', '0')))


def set_default_device(device):
    """Device used by the drop-in classes of this process (one process per GPU)."""
    global _default_device
    _default_device = int(device)


def default_handle(device=None):
    """Process-wide handle per device, shared by the drop-in classes (work space is reused)."""
    if device is None:
        device = _default_device
    h = _default.get(device)
    if h is None:
        h = _default[device] = Handle(device)
    return h


# ---- Laplace paths (attached to Handle below to keep the class body readable) -----------------
def _laplace_fit(self, entry, args, max_iter, f0):
    """Calls gpb_pref_laplace / gpb_gpc_laplace: `args` are the arguments before use_f0, the out-parameters follow.
    A factorisation that fails for every jitter or inside the loop (info > 0) raises LinAlgError."""
    f = np.zeros(self.n) if f0 is None else as_f64(f0).reshape(-1).copy()
    lml = C.c_double()
    iters = C.c_int32()
    info = C.c_int32()
    jit = C.c_double()
    trace = np.zeros((int(max_iter), 2))
    rc = entry(self.h, *args, 0 if f0 is None else 1, _dp(f), C.byref(lml), C.byref(iters), _dp(trace), C.byref(jit),
               C.byref(info))
    if rc != 0 and info.value > 0:
        raise np.linalg.LinAlgError(self.lib.gpb_last_error(self.h).decode())
    self.check(rc)
    return f, lml.value, iters.value, trace[:iters.value].copy(), jit.value


def _pref_laplace(self, uvi, y, khyp, sigma=1.0, delta_f=1e-6, max_iter=1000, grad_mode=0, f0=None):
    """PreferenceGaussianProcess.calc_laplace on the device: returns (f (n,), lml, iters, trace, jitter)."""
    uvi = np.ascontiguousarray(uvi, dtype=np.int64).reshape(-1, 2)
    y = as_f64(y).reshape(-1)
    khyp = self._khyp(khyp, extra=1)
    P = uvi.shape[0]
    assert y.shape[0] == P
    return _laplace_fit(self, self.lib.gpb_pref_laplace, (uvi.ctypes.data_as(c_lp), _dp(y), P, _dp(khyp), float(sigma),
                                                          float(delta_f), int(max_iter), int(grad_mode)), max_iter, f0)


def _pref_derivatives(self, uvi, y, f, sigma=1.0, grad_mode=0):
    uvi = np.ascontiguousarray(uvi, dtype=np.int64).reshape(-1, 2)
    y = as_f64(y).reshape(-1)
    f = as_f64(f).reshape(-1)
    n = f.shape[0]
    W = np.empty((n, n))
    g = np.empty(n)
    self.check(self.lib.gpb_pref_derivatives(self.h, uvi.ctypes.data_as(c_lp), _dp(y), uvi.shape[0], n, _dp(f),
                                             float(sigma), int(grad_mode), _dp(W), _dp(g)))
    return W, g


def _gpc_laplace(self, y, khyp, link=0, delta_f=1e-6, max_iter=100, f0=None):
    y = as_f64(y).reshape(-1)
    khyp = self._khyp(khyp, extra=1)
    return _laplace_fit(self, self.lib.gpb_gpc_laplace, (_dp(y), _dp(khyp), int(link), float(delta_f), int(max_iter)),
                        max_iter, f0)


def _gpc_predict(self, Z):
    Z = as_f64(Z)
    Z = Z.reshape(len(Z), -1)
    m = Z.shape[0]
    mu, var, p = np.empty(m), np.empty(m), np.empty(m)
    self.check(self.lib.gpb_gpc_predict(self.h, _dp(Z), m, _dp(mu), _dp(var), _dp(p)))
    return mu, var, p


def _gpc_evidence_grad(self):
    """(lml, grad) at the mode of the last gpc_laplace, whose loop must have converged: lml is the value gpc_laplace
    returned and grad is d lml / d [log l_1..log l_d, log sf] with the fit's jitter held fixed (opt-in, not in the
    reference)."""
    v = np.empty(1)
    g = np.empty(self.d + 1)
    self.check(self.lib.gpb_gpc_evidence_grad(self.h, _dp(v), _dp(g)))
    return float(v[0]), g


def _pref_evidence(self):
    """R&W eq. 3.32 at the mode of the last pref_laplace (opt-in, not in the reference)."""
    v = np.empty(1)
    self.check(self.lib.gpb_pref_evidence(self.h, _dp(v)))
    return float(v[0])


def _pref_evidence_grad(self):
    """(evidence, grad) at the mode of the last pref_laplace, which must have run with grad_mode=1: grad is
    d evidence / d [log l_1..log l_d, log sf, log sigma] with the fit's jitter held fixed (opt-in, not in the reference)."""
    v = np.empty(1)
    g = np.empty(self.d + 2)
    self.check(self.lib.gpb_pref_evidence_grad(self.h, _dp(v), _dp(g)))
    return float(v[0]), g


def _pref_predict(self, Z, Zb=None):
    """Latent posterior at Z, or of f(Zb) - f(Z) plus the preference probability (opt-in, not in the reference)."""
    Z = as_f64(Z)
    Z = Z.reshape(len(Z), -1)
    m = len(Z)
    mean, var = np.empty(m), np.empty(m)
    if Zb is None:
        self.check(self.lib.gpb_pref_predict(self.h, _dp(Z), None, m, _dp(mean), _dp(var), None))
        return mean, var
    Zb = as_f64(Zb).reshape(m, -1)
    prob = np.empty(m)
    self.check(self.lib.gpb_pref_predict(self.h, _dp(Z), _dp(Zb), m, _dp(mean), _dp(var), _dp(prob)))
    return mean, var, prob


def _pref_log_marginal(self, uvi, y, f, iK, logdetK, sigma=1.0):
    uvi = np.ascontiguousarray(uvi, dtype=np.int64).reshape(-1, 2)
    y = as_f64(y).reshape(-1)
    f = as_f64(f).reshape(-1)
    iK = as_f64(iK)
    assert iK.shape == (len(f), len(f)) and len(y) == len(uvi)
    v = np.empty(1)
    self.check(self.lib.gpb_pref_log_marginal(self.h, uvi.ctypes.data_as(c_lp), _dp(y), len(uvi), len(f), _dp(f), _dp(iK),
                                              float(logdetK), float(sigma), _dp(v)))
    return float(v[0])


Handle.pref_log_marginal = _pref_log_marginal
Handle.pref_evidence = _pref_evidence
Handle.pref_evidence_grad = _pref_evidence_grad
Handle.pref_predict = _pref_predict
Handle.pref_laplace = _pref_laplace
Handle.pref_derivatives = _pref_derivatives
Handle.gpc_laplace = _gpc_laplace
Handle.gpc_predict = _gpc_predict
Handle.gpc_evidence_grad = _gpc_evidence_grad
