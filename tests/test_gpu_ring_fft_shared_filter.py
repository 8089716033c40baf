"""The one-CTA-per-SM persistent ring FFT (`pxm_ring_fft6_kernel`: two 4-warp groups on chain pairs, one chirp and one
filter spectrum in shared memory, paired 16-byte stores of the ring array) against the two-CTA kernel it replaces
(`pxm_ring_fft3_kernel`, debug FFT mode 4) bit for bit (`pytest -m gpu`).

Both run the same codelets in the same order on the same items; only where the tables live, which threads run which item
and the width of the stores differ, so any difference in the output is a bug.  Cases: the bench shape (L = 256,
B = 1.5, J_min = 2) at 64 and 65 chains (an odd count leaves the second group of the last chain pair of every ring block
without an item), the class-edge grids L = 257 and 513, a grid whose persistent groups are all M = 512, and three MYULA
iterations of 64 chains as the bench runs them (predictions carried as ring coefficients).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OLD_KERNEL = 4  # pxm_debug_set_fft_multipass: the two-CTA persistent kernel for Bluestein lengths 512 / 1024
WAVELET_OPS = ("synthesis", "synthesis_adjoint", "analysis", "analysis_adjoint")  # both directions of the ring FFT


@pytest.fixture(scope="module")
def torch_dev():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _under(mode, fn):
    from pxmcmc_b200 import _lib

    try:
        _lib.check(_lib.lib.pxm_debug_set_fft_multipass(mode))
        return fn()
    finally:
        _lib.check(_lib.lib.pxm_debug_set_fft_multipass(0))


def _crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def _assert_same(got, ref, what):
    for name in got:
        assert np.array_equal(got[name], ref[name]), f"{what} {name}: the default ring FFT differs from the two-CTA kernel"


@pytest.mark.parametrize("L,B,nb", [(256, 1.5, 64), (256, 1.5, 65), (257, 2.0, 64), (513, 2.0, 64)])
def test_wavelet_operators_default_equals_two_cta_kernel(torch_dev, L, B, nb):
    """the four wavelet operators (pixels -> ring coefficients and back) at the bench shape and the class edges"""
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D

    plan = D.WaveletPlan(L, B, 2, nb)  # not cached
    try:
        rng = np.random.default_rng(L * 100 + nb)
        X = {"synthesis": _crandn(rng, nb, plan.ncoefs), "synthesis_adjoint": _crandn(rng, nb, plan.npix),
             "analysis": _crandn(rng, nb, plan.npix), "analysis_adjoint": _crandn(rng, nb, plan.ncoefs)}
        X = {name: D.to_dev_c(x) for name, x in X.items()}

        def run():
            out = {name: D.to_host(getattr(plan, name)(X[name])) for name in WAVELET_OPS}
            torch_dev.cuda.synchronize()
            return out

        _assert_same(run(), _under(OLD_KERNEL, run), f"L={L} B={B} nb={nb}")
    finally:
        _lib.check(_lib.lib.pxm_wav_plan_destroy(plan.h))
        plan.h = None


@pytest.mark.parametrize("nb", [64, 65])
def test_sht_on_m512_grid_default_equals_two_cta_kernel(torch_dev, nb):
    """one ring grid of bandlimit 100 (n = 199, Bluestein length 512 only; 13 ring blocks per chain: wide enough for
    the persistent kernel), all four spin-0 SHTs"""
    from pxmcmc_b200 import device as D

    L = 100
    plan = D.ShtPlan.get(L, 0, nb)
    rng = np.random.default_rng(nb)
    flm = D.to_dev_c(_crandn(rng, nb, L * L))
    pix = D.to_dev_c(_crandn(rng, nb, L * (2 * L - 1)))

    def run():
        out = {"inverse": D.to_host(plan.inverse(flm)), "forward": D.to_host(plan.forward(pix)),
               "inverse_adjoint": D.to_host(plan.inverse_adjoint(pix)), "forward_adjoint": D.to_host(plan.forward_adjoint(flm))}
        torch_dev.cuda.synchronize()
        return out

    _assert_same(run(), _under(OLD_KERNEL, run), f"SHT L={L} nb={nb}")


def test_myula_iterations_default_equal_two_cta_kernel(torch_dev):
    """three MYULA iterations of 64 chains at the bench shape, from the same state and Philox streams"""
    torch = torch_dev
    from pxmcmc_b200 import device as D
    from pxmcmc_b200.forward import SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1

    L, B, J, nch = 256, 1.5, 2, 64
    rng = np.random.default_rng(256)
    data = _crandn(rng, L * (2 * L - 1))
    op = SphericalWaveletTransformOperator(data, 1.0, "synthesis", L, B, J, nchains=nch)
    prm = PxMCMCParams(nsamples=1, nburn=0, ngap=1, delta=1e-6, lmda=1e-6, mu=1.0, verbosity=0, track=[])
    reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, prm.lmda * prm.mu, L=L, B=B, J_min=J)
    X0 = D.to_dev_c(rng.laplace(size=(nch, op.nparams)))

    def run():
        m = MYULA(op, reg, prm, noise="device", nchains=nch, seed=1234, stream0=0).engine
        m.forward.fuse_ring = True
        X = X0.clone()
        P = m._initial_preds(X)
        assert m._ring_mode(), "the predictions are no longer carried as ring coefficients"
        for _ in range(3):
            X, P = m.iterate(X, P)
        torch.cuda.synchronize()
        return {"state": D.to_host(X), "predictions": D.to_host(m._pix(P))}

    _assert_same(run(), _under(OLD_KERNEL, run), "MYULA")
