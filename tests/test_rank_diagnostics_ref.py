"""CPU tests of the rank-normalised diagnostics: the numpy oracle (oracle/rank_diagnostics_ref.py) pinned against
hand-computed ranks and known statistical behaviour, its edge cases, and the refusals of the host layer and the C ABI
(argument checks that run before anything touches a device)."""
import numpy as np
import pytest
from scipy.special import ndtri

from oracle import diagnostics_ref as D
from oracle import rank_diagnostics_ref as K


def _ar1(rng, phi, m, n, k):
    e = rng.standard_normal((m, n, k))
    x = np.empty_like(e)
    x[:, 0] = e[:, 0] / np.sqrt(1 - phi ** 2)
    for t in range(1, n):
        x[:, t] = phi * x[:, t - 1] + e[:, t]
    return x


def test_hand_computed_2x6_with_ties():
    x = np.array([[1.0, 2, 2, 3, 5, 8], [2, 4, 4, 6, 7, 9]])
    # split series (first halves, then second halves): [1 2 2] [2 4 4] [3 5 8] [6 7 9]; pooled order
    # 1 | 2 2 2 | 3 | 4 4 | 5 6 7 8 9  -> average ranks 1, 3, 5, 6.5, 8 .. 12
    ranks = np.array([[1, 3, 3], [3, 6.5, 6.5], [5, 8, 11], [9, 10, 12]])
    assert np.array_equal(K.split(x), [[1, 2, 2], [2, 4, 4], [3, 5, 8], [6, 7, 9]])
    zb = ndtri((ranks - 0.375) / 12.25)
    assert np.array_equal(K.z_scale(K.split(x)), zb)
    # median 4 (mean of the 6th and 7th of 12); |x - 4| = [3 2 2] [2 0 0] [1 1 4] [2 3 5]:
    # 0 0 | 1 1 | 2 2 2 2 | 3 3 | 4 | 5 -> 1.5, 3.5, 6.5, 9.5, 11, 12
    franks = np.array([[9.5, 6.5, 6.5], [6.5, 1.5, 1.5], [3.5, 3.5, 11], [6.5, 9.5, 12]])
    zf = ndtri((franks - 0.375) / 12.25)
    assert np.array_equal(K.z_scale(K.split(np.abs(x - 4.0))), zf)

    def R(s):  # 4 series of 3
        means = s.mean(axis=1)
        B = 3 * np.sum((means - means.mean()) ** 2) / 3
        W = np.mean(np.sum((s - means[:, None]) ** 2, axis=1) / 2)
        return np.sqrt((B / W + 2) / 3)

    rhat, bulk, tail = K.column(x)
    assert np.isclose(rhat, max(R(zb), R(zf)), rtol=1e-14, atol=0)
    assert R(zb) > R(zf)
    # h = 3: Geyer's loop never runs (t = 1 < h - 3 fails), T = -1, rho_hat[0] = 1, tau = max(0, 1 / log10 12).
    # q05 = 1 + 0.55 (2 - 1) -> only the 1 lies below; q95 = 8.45 -> only the 9 lies above: neither indicator is constant
    assert np.isclose(bulk, 12 * np.log10(12), rtol=1e-14)
    assert np.isclose(tail, 12 * np.log10(12), rtol=1e-14)


def test_R_of_raw_split_chains_is_bda3_split_rhat():
    x = np.random.default_rng(1).standard_normal((5, 37, 6)) * np.linspace(0.5, 3, 6) + np.arange(6)
    x[3] += 0.4
    want = D.summarise(x)["rhat"]
    for j in range(6):
        assert abs(K.R(K.split(x[:, :, j])) - want[j]) < 1e-14


def test_iid_normal():
    rhat, bulk, tail = K.rank_diagnostics(np.random.default_rng(2).standard_normal((4, 1000, 8)))
    assert np.all(rhat < 1.01)
    assert np.all(np.abs(bulk / 4000 - 1) < 0.1), bulk
    assert np.all(np.abs(tail / 4000 - 1) < 0.2), tail


def test_ar1_bulk_ess():
    phi, m, n = 0.9, 4, 1000
    _, bulk, _ = K.rank_diagnostics(_ar1(np.random.default_rng(3), phi, m, n, 16))
    want = m * n * (1 - phi) / (1 + phi)
    assert np.all(np.abs(bulk / want - 1) < 0.3), bulk / want
    assert abs(np.mean(bulk) / want - 1) < 0.1


def test_unequal_variances_caught_by_the_folded_rank_rhat_only():
    x = np.random.default_rng(4).standard_normal((4, 1000, 6))
    x[1::2] *= 2.0  # equal means, variances 1 and 4
    assert np.all(D.summarise(x)["rhat"] < 1.01)
    assert np.all(K.rank_diagnostics(x)[0] > 1.05)


def test_offset_chain():
    x = np.random.default_rng(5).standard_normal((4, 1000, 6))
    x[2] += 3.0
    rhat = K.rank_diagnostics(x)[0]
    assert np.all(rhat > 1.3) and np.all(np.abs(rhat - 1.48) < 0.05), rhat


def test_edge_cases():
    rng = np.random.default_rng(6)
    # constant column: z constant -> W = B = 0 -> NaN R-hat; both ESS are M h
    rhat, bulk, tail = K.rank_diagnostics(np.full((3, 10, 1), 2.5))
    assert np.isnan(rhat[0]) and bulk[0] == 30 and tail[0] == 30
    # n = 3: NaN; n = 4: defined
    assert all(np.isnan(v).all() for v in K.rank_diagnostics(rng.standard_normal((5, 3, 2))))
    assert all(np.isfinite(v).all() for v in K.rank_diagnostics(rng.standard_normal((5, 4, 2))))
    # odd n: the middle sample of each chain is in no series (but in the median and the quantiles)
    x = rng.standard_normal((2, 5))
    assert np.array_equal(K.split(x), np.concatenate([x[:, :2], x[:, 3:]]))
    # NaN or +-inf: NaN in that column only
    x = rng.standard_normal((4, 20, 5))
    x[1, 7, 1], x[0, 0, 3], x[3, 19, 4] = np.nan, np.inf, -np.inf
    out = np.array(K.rank_diagnostics(x))
    assert np.all(np.isnan(out[:, [1, 3, 4]])) and np.all(np.isfinite(out[:, [0, 2]]))
    # one chain as a 2-D array is m = 1
    assert np.array_equal(np.array(K.rank_diagnostics(x[0, :, [0, 2]].T)), np.array(K.rank_diagnostics(x[:1, :, [0, 2]])))


def test_host_refusals_before_any_device_work():
    from pxmcmc_b200.diagnostics import rank_diagnostics

    with pytest.raises(TypeError):
        rank_diagnostics(np.zeros((2, 8, 3), dtype=complex))
    with pytest.raises(ValueError):
        rank_diagnostics(np.zeros((2, 2, 8, 3)))
    with pytest.raises(ValueError, match="16384"):
        rank_diagnostics(np.zeros((1, 16385, 2)))


def test_c_abi_argument_checks():
    from pxmcmc_b200._lib import lib

    assert lib.pxm_rank_diagnostics_scratch_doubles(8, 2048, 3) == 8 * 2048 * 3
    assert lib.pxm_rank_diagnostics_scratch_doubles(1, 16385, 1) == -1
    assert lib.pxm_rank_diagnostics_scratch_doubles(0, 4, 1) == -1
    assert lib.pxm_rank_diagnostics(None, 2, 8193, 1, 1, None, None, None, None, None) != 0
    assert b"16384" in lib.pxm_last_error()
    assert lib.pxm_rank_diagnostics(None, 2, 8, 4, 3, None, None, None, None, None) != 0  # ld < ncols
    assert b"leading dimension" in lib.pxm_last_error()
