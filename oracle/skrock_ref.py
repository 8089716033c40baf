"""CPU restatement of SK-ROCK as published (Abdulle, Almuslimani & Vilmart, SIAM/ASA JUQ 2018; used for imaging by
Pereyra, Vargas-Mieles & Zygalakis, SIAM J. Imaging Sci. 2020).  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

The reference codes its recursion differently (``pxmcmc_ref.skrock_coefs`` / ``skrock_step``, kept as coded): its
ratio is T_{j-1}(omega_0) / T_j(omega_1) where the scheme has T_j(omega_0), and it adds a scalar k_j = 1 and
subtracts K_{j-2} where the scheme has kappa_j K_{j-2}, kappa_j = 1 - nu_j.  This module is what
``SKROCK(scheme="published")`` is checked against.
"""
import numpy as np

from .pxmcmc_ref import cheb1der, chebyshev1, gradlogpi


def skrock_omegas(s, eta=0.05):
    w0 = 1 + eta / (s * s)
    return w0, chebyshev1(w0, s) / cheb1der(w0, s)


def stability_limit(s, eta=0.05):
    """(omega_0 + 1) / omega_1: on p in [0, this], |R(p)| = |T_s(omega_0 - omega_1 p) / T_s(omega_0)| <= 1, and
    |R| = 1 / T_s(omega_0) at its end; |R| then grows and passes 1 at 2 omega_0 / omega_1"""
    w0, w1 = skrock_omegas(s, eta)
    return (w0 + 1) / w1


def skrock_coefs_published(s, eta=0.05):
    """mu_1 = omega_1/omega_0, nu_1 = s omega_1/2, kappa_1 = s omega_1/omega_0; for j >= 2
    mu_j = 2 omega_1 T_{j-1}(omega_0)/T_j(omega_0), nu_j = 2 omega_0 T_{j-1}(omega_0)/T_j(omega_0), kappa_j = 1 - nu_j.
    Returns (omega_0, omega_1, mus, nus, kappas) indexed 0..s like ``pxmcmc_ref.skrock_coefs``."""
    w0, w1 = skrock_omegas(s, eta)
    mus, nus, ks = np.zeros(s + 1), np.zeros(s + 1), np.zeros(s + 1)
    mus[1], nus[1], ks[1] = w1 / w0, s * w1 / 2, s * w1 / w0
    for j in range(2, s + 1):
        r = chebyshev1(w0, j - 1) / chebyshev1(w0, j)
        mus[j], nus[j], ks[j] = 2 * w1 * r, 2 * w0 * r, 1 - 2 * w0 * r
    return w0, w1, mus, nus, ks


def _recursion(grad, delta, s, X, Z, eta=0.05):
    _, _, mus, nus, ks = skrock_coefs_published(s, eta)
    sq = np.sqrt(2 * delta)
    K = [X]
    if s >= 1:
        K.append(X + mus[1] * delta * grad(X + nus[1] * sq * Z) + ks[1] * sq * Z)
    for j in range(2, s + 1):
        K.append(mus[j] * delta * grad(K[j - 1]) + nus[j] * K[j - 1] + ks[j] * K[j - 2])
    return K[s]


def skrock_step_published(fwd, prior, delta, lmda, s, X, Z):
    """K_0 = X; K_1 = X + mu_1 delta grad log pi(X + nu_1 sqrt(2 delta) Z) + kappa_1 sqrt(2 delta) Z;
    K_j = mu_j delta grad log pi(K_{j-1}) + nu_j K_{j-1} + kappa_j K_{j-2}; returns K_s (grad log pi as
    ``pxmcmc_ref.gradlogpi``)"""
    return _recursion(lambda x: gradlogpi(fwd, prior, lmda, x), delta, s, X, Z)


def scalar_step(a, d, delta, s, eta=0.05):
    """(R, S) of one published step on the scalar Gaussian target grad log pi(x) = -a (x - d): the step is the affine
    map x' - d = R (x - d) + S xi, so its stationary law is N(d, S^2 / (1 - R^2)) when |R| < 1"""
    step = lambda x, z: _recursion(lambda y: -a * (y - d), delta, s, x, z, eta)  # noqa: E731
    c = step(d, 0.0)  # = d: the target's mode is a fixed point
    return step(d + 1.0, 0.0) - c, step(d, 1.0) - c
