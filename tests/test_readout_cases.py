"""The extended-precision read-out references of ``readout_cases`` against the float64 oracle (CPU only)."""

import numpy as np
import pytest

import readout_cases as rc
import variant_cases as vc
from bodge_b200 import kpm
from oracle import bdg_oracle as orc


@pytest.fixture(scope="module")
def case():
    indptr, indices, data, scale = rc.random_hermitian_bsr((4, 3, 2), 3)
    scale *= 1.01
    x0 = orc.rademacher(9, 4 * (len(indptr) - 1), np.arange(5))
    return indptr, indices, data, scale, x0


def test_longdouble_is_wider_than_float64():
    vc.longdouble_check()


def test_scalar_reference_is_the_block_reference(case):
    indptr, indices, data, scale, x0 = case
    a = rc.reference_readouts(rc.ScalarReference(indptr, indices, data, scale), x0, 40)[0]
    b = rc.reference_readouts(vc.Reference(indptr, indices, data, scale), x0, 40)[0]
    assert np.max(np.abs(a - b)) <= 1e-16 * np.max(np.abs(b[0]))
    real = rc.ScalarReference(indptr, indices, data.real.astype(complex), scale)
    assert real.real and real.start(x0).dtype == np.longdouble


def test_moments_match_the_oracle(case):
    indptr, indices, data, scale, x0 = case
    H = orc.to_scipy(indptr, indices, data)
    mu = rc.reference_readouts(rc.ScalarReference(indptr, indices, data, scale), x0, 300)[0]
    want = orc.cheb_moments(H, x0, 300, scale)
    assert mu.dtype == np.longdouble
    assert np.max(np.abs(mu.astype(np.float64) - want)) <= 1e-12 * np.max(np.abs(want[0]))


def test_local_terms_and_sums(case):
    indptr, indices, data, scale, x0 = case
    Ht = orc.to_scipy(indptr, indices, data).toarray() / scale
    rows, cols = np.array([0, 5, 5, 95]), np.array([0, 4, 4, 2])
    _, terms, t_max = rc.reference_readouts(rc.ScalarReference(indptr, indices, data, scale), x0, 1, local=(rows, cols, 7))
    T = [x0, Ht @ x0]
    while len(T) < 7:
        T.append(2 * Ht @ T[-1] - T[-2])
    assert np.max(np.abs(terms.astype(np.complex128) - np.array([t[rows, cols] for t in T]))) <= 1e-12
    assert abs(t_max - max(np.max(np.abs(t)) for t in T)) <= 1e-12
    coef = np.linspace(1.0, -0.5, 7)
    got, size = rc.local_sums(terms, coef)
    assert np.max(np.abs(got.astype(np.complex128) - sum(c * t[rows, cols] for c, t in zip(coef, T)))) <= 1e-12
    assert np.all(size >= np.abs(got))


def test_resolvent_and_contraction_match_the_oracle(case):
    indptr, indices, data, scale, x0 = case
    mu = orc.cheb_moments(orc.to_scipy(indptr, indices, data), x0, 400, scale)
    z = np.array([0.3 + 0.1j, -0.999 - 0.05j, 0.0 + 0.02j])
    w, pref = kpm.resolvent_weights(z)
    got, size = rc.resolvent(mu, w, pref)
    for c in range(mu.shape[1]):
        for e in range(len(z)):
            want = kpm.resolvent_diagonal(mu[:, c], z[e])
            assert abs(complex(got[c, e]) - want) <= 1e-12 * float(size[c, e])
    assert np.all(size >= np.abs(got))
    coef = np.random.default_rng(1).uniform(-1, 1, 400)
    out, size = rc.contract(mu, coef)
    assert np.allclose(out.astype(np.float64), coef @ mu, rtol=0, atol=1e-12 * float(np.max(size)))


def test_warp_sum_order():
    # lane 0: 1e16 then 1.0 (rounds back to 1e16), lane 1: 1.0, lane 2: -1e16; the butterfly gives (1e16 - 1e16) + 1.0
    v = np.array([1e16, 1.0, -1e16] + [0.0] * 29 + [1.0])
    assert rc.warp_sum(v) == 1.0
    assert rc.warp_sum(np.arange(100.0)) == 4950.0
    assert rc.warp_sum([2.5]) == 2.5


def test_moment_ratios():
    want = np.array([[4.0], [1.0], [0.5]], dtype=np.longdouble)
    got = want.astype(np.float64) + np.array([[0.0], [0.0], [3 * 4.0 * rc.EPS]])
    r = rc.moment_ratios(got, want)
    assert r[0, 0] == 0 and abs(float(r[2, 0]) - 1.0) < 1e-6
    assert rc.worst(r, 1) == 0 and rc.worst(r, 0) == rc.worst(r)
