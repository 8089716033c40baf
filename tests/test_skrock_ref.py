"""CPU tests of the published SK-ROCK restatement (oracle/skrock_ref.py): the coefficients are those of Abdulle,
Almuslimani & Vilmart (2018), one step on a scalar Gaussian target has the closed-form deterministic factor
T_s(omega_0 - omega_1 p) / T_s(omega_0), which is stable up to (omega_0 + 1) / omega_1 and a little beyond, and the
sampler reports that limit."""
import numpy as np
import pytest
from numpy.polynomial import chebyshev as C

from oracle import skrock_ref as S


def _T(x, k):
    return C.chebval(x, [0] * k + [1])


@pytest.mark.parametrize("s", [2, 3, 5, 10, 15])
def test_kappa_is_minus_the_chebyshev_ratio(s):
    w0, w1, mus, nus, ks = S.skrock_coefs_published(s)
    for j in range(2, s + 1):
        assert np.isclose(ks[j], 1 - nus[j], rtol=0, atol=1e-15)
        assert np.isclose(ks[j], -_T(w0, j - 2) / _T(w0, j), rtol=1e-13)
        assert np.isclose(mus[j], 2 * w1 * _T(w0, j - 1) / _T(w0, j), rtol=1e-14)
    assert (mus[1], nus[1], ks[1]) == (w1 / w0, s * w1 / 2, s * w1 / w0)


@pytest.mark.parametrize("s", [1, 3, 5, 10, 15])
def test_scalar_step_is_the_chebyshev_stability_polynomial(s):
    w0, w1 = S.skrock_omegas(s)
    lim = S.stability_limit(s)
    for ad in np.concatenate([np.linspace(0, lim, 57), [1e-3, 0.1, 1.0, 10.0]]):
        R, _ = S.scalar_step(1.0, 0.0, ad, s)
        assert abs(R - _T(w0 - w1 * ad, s) / _T(w0, s)) < 1e-13


@pytest.mark.parametrize("s", [1, 3, 5, 10, 15])
def test_stable_up_to_the_limit_and_not_beyond(s):
    """|R| <= 1 on [0, (omega_0 + 1)/omega_1], with |R| = 1/T_s(omega_0) at its end; beyond it |R| grows and passes 1
    at 2 omega_0/omega_1, (omega_0 - 1)/omega_1 further (2.5e-4 of the limit at s = 10)"""
    w0, w1 = S.skrock_omegas(s)
    lim = S.stability_limit(s)
    Rs = np.array([S.scalar_step(1.0, 0.0, p, s)[0] for p in np.linspace(0, lim, 2001)])
    assert np.abs(Rs).max() <= 1 + 1e-12
    assert abs(Rs[-1]) == pytest.approx(1 / _T(w0, s), rel=1e-12)
    edge = 2 * w0 / w1
    assert edge - lim == pytest.approx((w0 - 1) / w1, rel=1e-9)
    assert abs(S.scalar_step(1.0, 0.0, edge * (1 - 1e-9), s)[0]) <= 1
    assert abs(S.scalar_step(1.0, 0.0, edge * (1 + 1e-6), s)[0]) > 1
    assert np.isclose([S.stability_limit(3), S.stability_limit(5), S.stability_limit(10)], [17.4, 48.4, 193.6],
                      atol=0.05).all()


def test_mode_is_a_fixed_point():
    """with Z = 0 the target's mean d is left where it is, for every coordinate's stiffness"""
    a, d = np.array([1.0, 40.0, 150.0]), np.array([0.3, -2.0, 5.0])
    for s, delta in ((3, 0.05), (10, 0.15)):
        x = S._recursion(lambda y: -a * (y - d), delta, s, d.copy(), np.zeros(3))
        assert np.allclose(x, d, rtol=0, atol=1e-13)
        R, _ = S.scalar_step(a, d, delta, s)
        assert (np.abs(R) < 1).all()
    # small a delta: the stationary variance S^2 / (1 - R^2) tends to the target's 1/a
    R, Sx = S.scalar_step(1.0, 0.0, 1e-3, 10)
    assert np.isclose(Sx ** 2 / (1 - R ** 2), 1.0, rtol=1e-3)


def test_step_matches_the_scalar_map():
    """skrock_step_published on a diagonal Gaussian (identity operators, T = 0) is the scalar map per coordinate"""
    from oracle import pxmcmc_ref as R

    n, lmda, delta, s = 6, 1e-3, 0.02, 5
    rng = np.random.default_rng(2)
    d = rng.standard_normal(n)
    sig = np.linspace(0.5, 2.0, n)
    t = R.IdentityTransform()
    op = R.ForwardOperator(d, sig, "synthesis", t, R.IdentityMeasurement(n, n), n)
    pr = R.L1("synthesis", t.inverse, t.inverse_adjoint, 0.0)
    X, Z = rng.standard_normal(n), rng.standard_normal(n)
    got = S.skrock_step_published(op, pr, delta, lmda, s, X, Z)
    # the prox term vanishes at T = 0; grad log pi = -invcov (x - d) (calc_gradg has no factor 1/2)
    Rm, Sm = S.scalar_step(1 / sig ** 2, d, delta, s)
    assert np.allclose(got, d + Rm * (X - d) + Sm * Z, rtol=1e-12, atol=1e-12)


def test_sampler_reports_the_limit():
    from pxmcmc_b200.forward import ForwardOperator
    from pxmcmc_b200.mcmc import SKROCK, PxMCMCParams
    from pxmcmc_b200.measurements import Identity
    from pxmcmc_b200.prior import L1
    from pxmcmc_b200.transforms import IdentityTransform

    d = np.arange(4.0)
    t = IdentityTransform()
    op = ForwardOperator(d, 0.1, "synthesis", t, Identity(4, 4), nparams=4)
    reg = L1("synthesis", t.inverse, t.inverse_adjoint, 0.0)
    for s in (1, 3, 10):
        prm = PxMCMCParams(s=s, nsamples=2, verbosity=0)
        m = SKROCK(op, reg, prm, scheme="published")
        assert m.scheme == "published"
        assert m.stability_limit == pytest.approx(S.stability_limit(s), rel=1e-15)
        _, _, mus, nus, ks = S.skrock_coefs_published(s)
        assert np.allclose(m.mus, mus, rtol=1e-15) and np.allclose(m.nus, nus, rtol=1e-15)
        assert np.allclose(m.ks, ks, rtol=1e-13, atol=1e-15)
        ref = SKROCK(op, reg, prm)
        assert ref.scheme == "reference" and np.isnan(ref.stability_limit)
        assert np.array_equal(ref.mus[:2], m.mus[:2]) and np.array_equal(ref.ks[:2], m.ks[:2])
    with pytest.raises(ValueError):
        SKROCK(op, reg, PxMCMCParams(s=3, nsamples=2, verbosity=0), scheme="coded")
    with pytest.raises(AttributeError):
        m.stability_limit = 1.0
