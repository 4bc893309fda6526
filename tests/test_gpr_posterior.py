"""CPU checks of the oracle side of the joint posterior and the posterior samples (gpb_gpr_predict_full /
gpb_gpr_sample): the Philox4x32-10 restatement against the Random123 known answers, the moments of its normals,
and predict_full_chol against predict_chol and the reference's inv()-based form."""
import numpy as np
import pytest

from oracle import gpr_oracle
from tests import _posterior_oracle as po


@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
])
def test_philox_known_answers(ctr, key, want):
    got = po.philox4x32_10(np.array(ctr, dtype=np.uint64), np.array(key, dtype=np.uint64))
    assert [int(v) for v in got] == want


def test_philox_normals_layout():
    e = po.philox_normals(12345, 3, 7)
    assert e.shape == (3, 7)
    # the draws of the first points do not depend on how many points follow, nor those of the first samples on nsamp
    np.testing.assert_array_equal(po.philox_normals(12345, 3, 4), e[:, :4])
    np.testing.assert_array_equal(po.philox_normals(12345, 2, 7), e[:2])
    assert not np.array_equal(po.philox_normals(12346, 3, 7), e)
    # a pair shares one Philox block: e[s, 2p]^2 + e[s, 2p + 1]^2 = -2 ln u1 with u1 from words 0 and 1
    x = po.philox4x32_10(np.array([1, 0, 2, 0], dtype=np.uint64),
                         np.array([12345, 0], dtype=np.uint64)).astype(np.uint64)
    u1 = float(((int(x[0]) | (int(x[1]) << 32)) >> 11) + 1) * 2.0 ** -53
    assert e[2, 2] ** 2 + e[2, 3] ** 2 == pytest.approx(-2.0 * np.log(u1), rel=1e-14)


def test_philox_normals_moments():
    e = po.philox_normals(2024, 1000, 1000).ravel()
    n = e.size
    assert abs(e.mean()) < 6.0 / np.sqrt(n)
    assert abs(e.var() - 1.0) < 6.0 * np.sqrt(2.0 / n)


@pytest.mark.parametrize("kind", ["SE", "Matern32", "Matern52"])
def test_predict_full_chol_diagonal_is_predict_chol(kind):
    rng = np.random.default_rng(3)
    x = rng.random((40, 2))
    y = np.sin(4 * x[:, 0]) + 0.1 * rng.standard_normal(40)
    z = rng.random((25, 2))
    lh = np.log([0.4, 0.7, 1.3, 0.1])
    fz, cov = po.predict_full_chol(lh, x, y, z, kind)
    mu, var = gpr_oracle.predict_kind(lh, x, y, z, kind)
    np.testing.assert_allclose(fz, mu, rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(np.diag(cov), var, rtol=0, atol=1e-12)
    _, covn = po.predict_full_chol(lh, x, y, z, kind, noisy=True)
    np.testing.assert_allclose(covn - cov, 0.1 ** 2 * np.eye(25), rtol=0, atol=1e-15)


def test_predict_full_chol_matches_reference_form():
    rng = np.random.default_rng(4)
    x = rng.random((30, 1)) * 5
    y = np.cos(x[:, 0])
    z = rng.random((12, 1)) * 5
    lh = np.log([1.0, 1.0, 0.3])               # cond(K) ~ 1e3
    _, cov = po.predict_full_chol(lh, x, y, z)
    Kxz = gpr_oracle.kxz(lh, x, z)
    ref = gpr_oracle.kxz(lh, z, z) - Kxz.T @ np.linalg.inv(gpr_oracle.kxx(lh, x)) @ Kxz
    np.testing.assert_allclose(cov, ref, rtol=0, atol=1e-12)
