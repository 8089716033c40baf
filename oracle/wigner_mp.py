"""Arbitrary-precision Wigner d^l_{mn}(theta) by Wigner's explicit sum.  TEST INFRASTRUCTURE ONLY.

The device builds its Legendre tables with a three-term recurrence in l (pxmcmc_b200/csrc/pxm_wigner.cuh) and
oracle/ssht_ref.py expands d^l through d^l(pi/2) in double precision; this module shares neither route:

    d^l_{mn}(theta) = sum_k (-1)^(k-n+m) sqrt((l+m)! (l-m)! (l+n)! (l-n)!) / ((l+n-k)! k! (l-m-k)! (k-n+m)!)
                      * cos(theta/2)^(2l-2k+n-m) sin(theta/2)^(2k-n+m)

(the convention of ssht_ref.wigner_d_explicit), with exact integer factorials and mpmath at a precision that covers
the sum's cancellation: its terms exceed the result by up to about 2^(2l), so l = 1023 is evaluated with ~660 digits.

The colatitude is exact: theta = pi p / q for an integer pair (the MW rings, theta_t = pi (2t+1) / (2L-1)), or given
by the rational sin^2(theta/2) (the HEALPix rings, whose z = cos(theta) is rational).  Values are returned as mpf, so a
caller can tell a true magnitude below DBL_MIN from zero.
"""
from fractions import Fraction
from math import factorial, isqrt

import mpmath


def _dps(l):
    return int(0.61 * l) + 40


def _sign(e):
    return -1 if e & 1 else 1


def _sum(l, m, n, sh, ch):
    """the explicit sum at the current mpmath precision, sh = sin(theta/2), ch = cos(theta/2) (mpf)"""
    if not (abs(m) <= l and abs(n) <= l):
        raise ValueError(f"need |m|, |n| <= l (l={l}, m={m}, n={n})")
    k0, k1 = max(0, n - m), min(l + n, l - m)
    pref = mpmath.sqrt(mpmath.mpf(factorial(l + m) * factorial(l - m) * factorial(l + n) * factorial(l - n)))
    if sh == 0 or ch == 0:  # a pole: only the term whose vanishing power is zero survives (0^0 = 1)
        tot = mpmath.mpf(0)
        for k in range(k0, k1 + 1):
            a, b = 2 * l - 2 * k + n - m, 2 * k - n + m
            if (a and ch == 0) or (b and sh == 0):
                continue
            den = factorial(l + n - k) * factorial(k) * factorial(l - m - k) * factorial(k - n + m)
            tot += _sign(k - n + m) * ch ** a * sh ** b / den
        return pref * tot
    # Horner in x = tan^2(theta/2): term_{k+1} / term_k = -(l+n-k)(l-m-k) / ((k+1)(k+1-n+m)) x
    x = (sh / ch) ** 2
    acc = mpmath.mpf(1)
    for k in range(k1 - 1, k0 - 1, -1):
        acc = 1 - acc * x * ((l + n - k) * (l - m - k)) / ((k + 1) * (k + 1 - n + m))
    den0 = factorial(l + n - k0) * factorial(k0) * factorial(l - m - k0) * factorial(k0 - n + m)
    a0, b0 = 2 * l - 2 * k0 + n - m, 2 * k0 - n + m
    return _sign(k0 - n + m) * pref / den0 * ch ** a0 * sh ** b0 * acc


def wigner_d(l, m, n, p, q):
    """d^l_{mn}(pi p / q) for integers 0 <= p <= q, q > 0 (mpf, ~40 significant digits or better)"""
    if not (q > 0 and 0 <= p <= q):
        raise ValueError("theta = pi p / q must lie in [0, pi]")
    with mpmath.workdps(_dps(l)):
        half = mpmath.mpf(p) / (2 * q)  # theta / (2 pi)
        if p == 0 or p == q:  # the poles: exact zeros, so that the sum keeps its one surviving term
            sh, ch = mpmath.mpf(p // q), mpmath.mpf(1 - p // q)
        else:
            sh, ch = mpmath.sinpi(half), mpmath.cospi(half)
        return +_sum(l, m, n, sh, ch)


def wigner_d_sin2(l, m, n, s2):
    """d^l_{mn}(theta) with sin^2(theta/2) = s2 given exactly (a Fraction in [0, 1]); mpf"""
    s2 = Fraction(s2)
    if not 0 <= s2 <= 1:
        raise ValueError("sin^2(theta/2) must lie in [0, 1]")
    with mpmath.workdps(_dps(l)):
        sh = _sqrt_fraction(s2)
        ch = _sqrt_fraction(1 - s2)
        return +_sum(l, m, n, sh, ch)


def _sqrt_fraction(f):
    if f == 0:
        return mpmath.mpf(0)
    rn, rd = isqrt(f.numerator), isqrt(f.denominator)
    if rn * rn == f.numerator and rd * rd == f.denominator:
        return mpmath.mpf(rn) / rd
    return mpmath.sqrt(mpmath.mpf(f.numerator) / f.denominator)


def healpix_sin2_half(nside, i):
    """sin^2(theta_i / 2) of HEALPix ring i = 1 ... 4 nside - 1, exactly: (1 - z_i) / 2 with the rational z_i of the
    polar caps (1 - |z| = i'^2 / (3 nside^2)) and of the equatorial belt (z = 4/3 - 2 i / (3 nside))"""
    if not 1 <= i <= 4 * nside - 1:
        raise ValueError("ring index out of range")
    if i < nside:
        return Fraction(i * i, 6 * nside * nside)
    if i <= 3 * nside:
        return Fraction(2 * i - nside, 6 * nside)
    ip = 4 * nside - i
    return 1 - Fraction(ip * ip, 6 * nside * nside)
