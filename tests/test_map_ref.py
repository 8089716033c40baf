"""CPU tests of the MAP oracle (oracle/map_ref.py): the dense matrix of the data-fidelity gradient's linear part is
Hermitian positive semi-definite, the numpy FISTA with step 1 / lambda_max reaches the minimiser's fixed-point condition,
and MYULA's stability limit is where the scalar recursion's factor leaves [-1, 1]."""
import numpy as np
import pytest
from scipy import sparse

from conftest import golden
from oracle import map_ref as M
from oracle import pxmcmc_ref as R

L, B, J = 10, 2.0, 2
NPIX = L * (2 * L - 1)


def _wavelet_case(sig):
    t = R.WaveletTransform(L, B, J)
    data = np.random.default_rng(0).standard_normal(NPIX)
    return R.ForwardOperator(data, sig, "synthesis", t, R.IdentityMeasurement(NPIX, NPIX), t.ncoefs), t


@pytest.fixture(scope="module")
def scalar_case():
    op, t = _wavelet_case(0.3)
    return op, t, M.dense_operator(op)


class _Dense:
    """gradg(x) = M x - b from the dense oracle matrix (b = -gradg(0)): the same map as the operator, fast enough to run
    FISTA to convergence on the CPU"""

    def __init__(self, op, Mx):
        self.Mx, self.b = Mx, -M.gradg(op, np.zeros(op.nparams))

    def forward(self, x):
        return x

    def calc_gradg(self, x):
        return self.Mx @ x - self.b


def _psd(Mx):
    assert np.abs(Mx - Mx.conj().T).max() <= 1e-13 * np.abs(Mx).max()
    ev = np.linalg.eigvalsh(Mx)
    assert ev[0] >= -1e-12 * ev[-1] and ev[-1] > 0
    return ev


def test_dense_operator_is_hermitian_psd(scalar_case):
    op, t, Mx = scalar_case
    ev = _psd(Mx)
    # <x, M x> = |IC^(1/2) Phi Psi x|^2
    x = np.random.default_rng(1).standard_normal(op.nparams)
    ic = op.invcov
    assert np.isclose(np.vdot(x, Mx @ x).real, np.sum(ic * np.abs(op.forward(x)) ** 2), rtol=1e-12)
    assert np.isclose(ev[-1], 1 / 0.3 ** 2 * np.linalg.eigvalsh(M.dense_operator(_wavelet_case(1.0)[0]))[-1], rtol=1e-10)


def test_dense_operator_path_integral_is_hermitian_psd():
    g = golden("ref_skrock_L10.npz")
    Lg, Bg, Jg = int(g["L"]), float(g["B"]), int(g["J_min"])
    A = sparse.csr_matrix((g["A_data"], g["A_indices"], g["A_indptr"]), shape=tuple(g["A_shape"]))
    t = R.WaveletTransform(Lg, Bg, Jg)
    op = R.ForwardOperator(g["data"], g["sig_d"], "synthesis", t, R.PathIntegral(A), t.ncoefs)
    _psd(M.dense_operator(op))


def test_numpy_fista_reaches_the_fixed_point(scalar_case):
    op, t, Mx = scalar_case
    lmda, mu, tol = 1e-4, 100.0, 1e-8
    prior = R.S2WaveletsL1("synthesis", t.inverse, t.inverse_adjoint, lmda * mu, L, B, J)
    step = 1.0 / np.linalg.eigvalsh(Mx)[-1]
    dense = _Dense(op, Mx)
    x0 = np.random.default_rng(2).laplace(size=op.nparams)
    # the first iterates agree with the wavelet operator itself
    a, b = M.fista(op, prior, lmda, step, x0, 5), M.fista(dense, prior, lmda, step, x0, 5)
    assert max(np.linalg.norm(u - v) / np.linalg.norm(v) for u, v in zip(a, b)) < 1e-11
    # FISTA as oracle/map_ref.fista states it, run until the relative change is below tol
    T = (step / lmda) * prior.T
    x = y = np.asarray(x0, dtype=complex)
    tau, rel, k = 1.0, np.inf, 0
    while rel >= tol and k < 100_000:
        xn = R.soft(y - step * dense.calc_gradg(y), T)
        tau_n = (1.0 + np.sqrt(1.0 + 4.0 * tau * tau)) / 2.0
        y = xn + ((tau - 1.0) / tau_n) * (xn - x)
        rel = np.linalg.norm(xn - x) / np.linalg.norm(xn)
        x, tau, k = xn, tau_n, k + 1
    assert rel < tol
    assert M.fixed_point_residual(op, prior, lmda, step, x) <= 10 * tol
    assert np.mean(x == 0) > 0.5  # the threshold is active: a sparse minimiser
    # F does not increase under further proximal-gradient steps from the minimiser
    F = M.objective(op, prior, mu, x)
    assert M.objective(op, prior, mu, M.ista(dense, prior, lmda, step, x, 100)) >= F - 1e-10 * abs(F)


def test_myula_stability_limit_matches_the_scalar_recursion():
    from pxmcmc_b200.mcmc import MYULA

    lim = MYULA.stability_limit
    a, lmda = 3.0, 0.5
    lip = a + 1 / lmda  # gradg and the Moreau-Yosida term (the threshold zeroes x)
    assert M.myula_factor(a, lmda, lim / lip) == pytest.approx(-1.0, abs=1e-14)
    assert abs(M.myula_factor(a, lmda, 0.999 * lim / lip)) < 1
    assert abs(M.myula_factor(a, lmda, 1.001 * lim / lip)) > 1
    for p in np.linspace(0.0, lim, 9):
        assert abs(M.myula_factor(a, lmda, p / lip)) <= 1 + 1e-14
    # no prior term (T = 0): the factor is 1 - delta a
    assert M.myula_factor(a, lmda, lim / a, T=0.0) == pytest.approx(-1.0, abs=1e-14)
