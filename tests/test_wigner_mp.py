"""The arbitrary-precision Wigner reference (oracle/wigner_mp.py) is itself right: the GPU tests compare the device
Legendre tables with it at L = 1024, so it must not carry a defect the comparison would then accept.  Then the host
compile of the library's recurrence against it at L = 1024, where the polar seeds underflow by thousands of decades."""
from fractions import Fraction
from math import pi

import mpmath
import numpy as np
import pytest

from oracle import healpix_ref, ssht_ref
from oracle import wigner_mp as W


def test_closed_form_at_small_l():
    """every (l, m, n) with l < 9 at three colatitudes against ssht_ref.wigner_d_explicit (double precision)"""
    for p, q in ((1, 17), (6, 13), (16, 17)):
        for l in range(9):
            for m in range(-l, l + 1):
                for n in range(-l, l + 1):
                    ref = ssht_ref.wigner_d_explicit(l, m, n, pi * p / q)
                    assert abs(float(W.wigner_d(l, m, n, p, q)) - ref) < 1e-14, (l, m, n, p, q)


@pytest.mark.parametrize("l", [0, 1, 2, 7, 40, 1023])
def test_poles(l):
    """d^l_{mn}(0) = delta_{mn}, d^l_{mn}(pi) = (-1)^(l+m) delta_{m,-n}: the zeros exact, the ones to 1e-40"""
    ms = range(-l, l + 1) if l < 10 else (-l, -l + 1, -1, 0, 1, 2, l - 1, l)
    for m in ms:
        for n in ms:
            for (p, q), ref in (((0, 1), int(m == n)), ((1, 1), (-1) ** ((l + m) & 1) * int(m == -n)),
                                ((7, 7), (-1) ** ((l + m) & 1) * int(m == -n))):
                d = W.wigner_d(l, m, n, p, q)
                assert (d == 0) if ref == 0 else abs(d - ref) < 1e-40, (l, m, n, p, q, d)


@pytest.mark.parametrize("l,m,n,p,q", [(1023, 3, -2, 5, 2047), (1023, 1023, 0, 1, 2047), (1023, -511, 2, 1023, 2047),
                                       (700, 250, 1, 3, 7), (1023, 1022, -2, 2045, 2047), (64, -64, 64, 1, 3)])
def test_symmetries(l, m, n, p, q):
    """d_{mn} = (-1)^(m-n) d_{nm} = d_{-n,-m}, to 1e-35 relative, including values far below DBL_MIN"""
    a, b, c = W.wigner_d(l, m, n, p, q), W.wigner_d(l, n, m, p, q), W.wigner_d(l, -n, -m, p, q)
    assert a != 0
    with mpmath.workdps(60):  # (mpf arithmetic rounds to the working precision)
        b = (-1) ** ((m - n) & 1) * b
        assert abs(a - b) <= 1e-35 * abs(a) and abs(a - c) <= 1e-35 * abs(a)


def test_unitarity_at_l_1023():
    """sum_n d^l_{mn}(theta)^2 = 1 at l = 1023, m = 0 (the longest sums, the deepest cancellation), to 1e-30"""
    l = 1023
    with mpmath.workdps(50):
        tot = mpmath.fsum(W.wigner_d(l, 0, n, 3, 7) ** 2 for n in range(-l, l + 1))
        assert abs(tot - 1) < mpmath.mpf(10) ** -30


def test_healpix_colatitudes_are_exact():
    """the rational sin^2(theta/2) of every HEALPix ring equals (1 - z) / 2 of the oracle's ring table, and the
    rational-colatitude and pi p / q forms agree where both apply (theta = pi/3, pi/2, 2pi/3)"""
    nside = 8
    for i, (_, _, _, z) in enumerate(healpix_ref.ring_table(nside), start=1):
        assert abs(float(W.healpix_sin2_half(nside, i)) - (1 - z) / 2) < 2e-16
    assert W.healpix_sin2_half(nside, 2 * nside) == Fraction(1, 2)
    for s2, (p, q) in ((Fraction(1, 4), (1, 3)), (Fraction(1, 2), (1, 2)), (Fraction(3, 4), (2, 3))):
        for l, m, n in ((9, 2, -2), (300, 17, 0), (301, 301, 2)):
            a, b = W.wigner_d_sin2(l, m, n, s2), W.wigner_d(l, m, n, p, q)
            with mpmath.workdps(60):
                assert b != 0 and abs(a - b) <= 1e-35 * abs(b), (l, m, n, s2)


# ------------------------------------------------------------------ the library's host-compiled recurrence, L = 1024
HOST_ROWS = [  # (ring, m, spin): both polar rings, theta = pi, the rings on either side of theta = pi/2
    (0, 1023, 0), (0, 0, 0), (1, -700, 2), (1023, 1, 0), (1023, -2, 2), (1023, 1023, -2), (1022, 1023, 0),
    (511, 1023, 2), (512, -1023, 0), (512, 3, 2),
    (96, 511, 0), (96, -511, 2),  # seed below e^-600 that grows back past 1e-100: the 2^300 rescale with an exponent
]


@pytest.mark.parametrize("ring,m,spin", HOST_ROWS)
def test_host_recurrence_at_l_1024_against_explicit_sum(ring, m, spin):
    """Lambda^{m,s}_l(theta_t) from pxm_debug_wigner_row_host (the same recurrence the device tables run) at a dozen
    degrees of one row: within 1e-12 sqrt((2l+1)/4pi), and zero or subnormal where the true value is below DBL_MIN
    (theta = pi rows are exactly zero but for m = -n)"""
    from pxmcmc_b200 import _lib

    L = 1024
    row = _lib.wigner_row_host(L, ring, m, spin, L)
    l0 = max(abs(m), abs(spin))
    ls = sorted(l for l in {l0, l0 + 1, l0 + 2, (l0 + L) // 2, L - 3, L - 2, L - 1} if l0 <= l < L)
    for l in ls:
        d = W.wigner_d(l, m, -spin, 2 * ring + 1, 2 * L - 1)
        with mpmath.workdps(30):
            ref = (-1) ** (abs(spin) & 1) * mpmath.sqrt(mpmath.mpf(2 * l + 1) / (4 * mpmath.pi)) * d
        if abs(ref) < np.finfo(np.float64).tiny:
            assert abs(row[l]) < np.finfo(np.float64).tiny, (l, float(abs(ref)), row[l])
        else:  # absolute bar; relative too for tiny values before the row's turning point (the exponent tracking)
            bar = 1e-12 * np.sqrt((2 * l + 1) / (4 * np.pi))
            polar = (l + 0.5) * np.sin(np.pi * (2 * ring + 1) / (2 * L - 1)) < max(abs(m), abs(spin))
            if 1e-280 < abs(ref) < 1e-30 and polar:
                bar = min(bar, 1e-10 * float(abs(ref)))
            assert abs(row[l] - float(ref)) <= bar, (l, float(ref), row[l])
    assert np.all(row[:l0] == 0)
