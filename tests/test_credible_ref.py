"""CPU tests of the index arithmetic behind the streaming credible intervals (pxm_credible_*, DESIGN.md 7b): numpy's
linear quantiles at alpha / 2 and 1 - alpha / 2 of N values, restated from the K_lo = min(lo_a + 2, N) smallest and the
K_hi = N - lo_b largest values alone, as the device heaps hold them, equal np.quantile bit for bit."""
import numpy as np
import pytest

from pxmcmc_b200.diagnostics import CredibleIntervals, credible_tails


def _lerp(a, b, t):
    """numpy's _lerp (quantile method "linear")"""
    d = b - a
    return b - d * (1 - t) if t >= 0.5 else a + d * t


def from_tails(x, alpha):
    """(lower, upper) of the columns of x [N, E] from the bounded tails only"""
    N, lo_a, g_a, lo_b, g_b = credible_tails(x.shape[0], alpha)
    klo, khi = min(lo_a + 2, N), N - lo_b
    s = np.sort(x, axis=0)
    small, large = s[:klo], s[N - khi:]  # the K_lo smallest, the K_hi largest (ascending)
    # the heaps' roots and larger children: x(K_lo - 1), x(K_lo - 2); x(lo_b), x(lo_b + 1)
    xa = small[-2] if lo_a != min(lo_a + 1, N - 1) else small[-1]
    ra = small[-1]
    rb = large[0]
    xb = large[1] if min(lo_b + 1, N - 1) != lo_b else large[0]
    with np.errstate(invalid="ignore"):
        lower = np.array([_lerp(a, b, g_a) for a, b in zip(xa, ra)])
        upper = np.array([_lerp(a, b, g_b) for a, b in zip(rb, xb)])
    nan = np.isnan(x).any(axis=0)
    lower[nan] = np.nan
    upper[nan] = np.nan
    return lower, upper


ALPHAS = [0.001, 0.01, 0.05, 0.1, 0.3, 0.5, 0.9, 0.99, 0.999]


@pytest.mark.parametrize("alpha", ALPHAS)
def test_tails_give_numpy_quantiles(alpha):
    rng = np.random.default_rng(int(alpha * 1e4))
    for N in list(range(1, 70)) + [99, 100, 101, 257, 1000, 1001, 12800]:
        x = rng.standard_normal((N, 7))
        x[:, 1] = np.floor(x[:, 1] * 2)  # heavy ties
        x[:, 2] = np.where(rng.uniform(size=N) < 0.5, 0.0, -0.0)  # signed zeros only
        x[:, 3] = rng.standard_cauchy(N)
        x[:, 4] = np.where(rng.uniform(size=N) < 0.1, np.inf, x[:, 4])
        x[:, 5] = np.where(rng.uniform(size=N) < 0.1, -np.inf, x[:, 5])
        if N > 3:
            x[N // 3, 6] = np.nan
        lo, hi = from_tails(x, alpha)
        with np.errstate(invalid="ignore"):
            ref_lo, ref_hi = np.quantile(x, alpha / 2, axis=0), np.quantile(x, 1 - alpha / 2, axis=0)
        assert np.array_equal(lo, ref_lo, equal_nan=True), (N, alpha)
        assert np.array_equal(hi, ref_hi, equal_nan=True), (N, alpha)


def test_tail_sizes():
    """the bound the heaps are sized by: about alpha / 2 of N per tail, never more than N, at least one"""
    for N in (1, 2, 3, 10, 12800, 64000):
        for alpha in ALPHAS:
            _, lo_a, _, lo_b, _ = credible_tails(N, alpha)
            klo, khi = min(lo_a + 2, N), N - lo_b
            assert 1 <= klo <= N and 1 <= khi <= N
            assert klo <= alpha / 2 * (N - 1) + 2 and khi <= alpha / 2 * (N - 1) + 2
    assert credible_tails(12800, 0.05)[1] + 2 == 321  # the bench shape: 64 chains x 200 samples


def test_credible_intervals_fields():
    ci = CredibleIntervals(0.1, 3, 5, np.array([-1.0, 0.5]), np.array([2.0, 0.5]))
    assert ci.npooled == 15 and ci.alpha == 0.1
    assert np.array_equal(ci.range, np.array([3.0, 0.0]))
