"""Reference side of the joint posterior covariance and the posterior samples of GP regression (gpb_gpr_predict_full,
gpb_gpr_sample): test infrastructure, like oracle/, on top of oracle/gpr_oracle.py.  Neither is in the reference,
which keeps only the diagonal of Kzx inv(K) Kxz (GPr.py:50)."""
import numpy as np

from oracle import gpr_oracle


def predict_full_chol(log_hyp, x, y, z, kind='SE', noisy=False):
    """(fz, Kzz - Kzx K^-1 Kxz (+ sn2 I if noisy)) through the Cholesky factor of K, like predict_chol."""
    from scipy.linalg import cho_solve, solve_triangular
    K = gpr_oracle.kxx_kind(log_hyp, x, kind)
    Ks = gpr_oracle.kxz_kind(log_hyp, x, z, kind)
    L = np.linalg.cholesky(K)
    alpha = cho_solve((L, True), np.asarray(y, dtype=float).reshape(-1))
    V = solve_triangular(L, Ks, lower=True)
    _, sf2, sn2 = gpr_oracle.split_hyp(log_hyp)
    Kzz = gpr_oracle.kxz_kind(log_hyp, z, z, kind)
    np.fill_diagonal(Kzz, sf2)                     # zero distance of a point to itself
    cov = Kzz - V.T @ V
    if noisy:
        cov = cov + sn2 * np.eye(len(cov))
    return Ks.T @ alpha, cov


PHILOX_M = (0xD2511F53, 0xCD9E8D57)
PHILOX_W = (0x9E3779B9, 0xBB67AE85)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11) on arrays: ctr (..., 4) and key (..., 2) of uint32 -> (..., 4) uint32.
    Products in uint64, so every operation is exact."""
    c = [np.asarray(ctr, dtype=np.uint64)[..., i] for i in range(4)]
    k = [np.asarray(key, dtype=np.uint64)[..., i] for i in range(2)]
    mask = np.uint64(0xFFFFFFFF)
    for r in range(10):
        if r:
            k = [(k[0] + np.uint64(PHILOX_W[0])) & mask, (k[1] + np.uint64(PHILOX_W[1])) & mask]
        p0 = np.uint64(PHILOX_M[0]) * c[0]
        p1 = np.uint64(PHILOX_M[1]) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k[0], p1 & mask, (p0 >> np.uint64(32)) ^ c[3] ^ k[1], p0 & mask]
    return np.stack(c, axis=-1).astype(np.uint32)


def philox_normals(seed, nsamp, m):
    """The standard normals gpb_gpr_sample draws, (nsamp, m): for sample s and pair p = i // 2, Philox4x32-10 with
    counter (p lo, p hi, s lo, s hi) and key (seed lo, seed hi); u1 = (((x0 | x1 << 32) >> 11) + 1) 2^-53,
    u2 = ((x2 | x3 << 32) >> 11) 2^-53; e[s, 2p] = sqrt(-2 ln u1) cos(2 pi u2), e[s, 2p + 1] = ... sin(2 pi u2)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    npair = (int(m) + 1) // 2
    s, p = np.meshgrid(np.arange(nsamp, dtype=np.uint64), np.arange(npair, dtype=np.uint64), indexing='ij')
    lo = np.uint64(0xFFFFFFFF)
    ctr = np.stack([p & lo, p >> np.uint64(32), s & lo, s >> np.uint64(32)], axis=-1)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64), ctr.shape[:-1] + (2,))
    x = philox4x32_10(ctr, key).astype(np.uint64)
    a = x[..., 0] | (x[..., 1] << np.uint64(32))
    b = x[..., 2] | (x[..., 3] << np.uint64(32))
    u1 = ((a >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    u2 = (b >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    r = np.sqrt(-2.0 * np.log(u1))
    t = 2 * np.pi * u2
    e = np.empty((int(nsamp), 2 * npair))
    e[:, 0::2] = r * np.cos(t)
    e[:, 1::2] = r * np.sin(t)
    return e[:, :int(m)]
