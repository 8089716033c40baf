"""GPU parity tests (run on the B200 box: `pytest -m gpu`).

Every test drives the CUDA path through the public Python classes, i.e. through
the C ABI of libpxmcmc_b200.so, and compares with
  * the committed fixtures produced by the unmodified reference (tests/golden), and
  * the CPU oracle (oracle/) on seeded inputs.
Tolerance: 1e-10 relative L2 in FP64 (BASELINE.json north_star); the prox
support / sign pattern and the real soft threshold must match exactly.
"""
import numpy as np
import pytest
from scipy import sparse

from conftest import golden, rel_l2
from oracle.philox_ref import philox_uniform as _philox_uniform

pytestmark = pytest.mark.gpu

TOL = 1e-10


@pytest.fixture(scope="module")
def px():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import pxmcmc_b200
    from pxmcmc_b200 import forward, mcmc, measurements, prior, sht, transforms, utils

    class NS:
        pass

    ns = NS()
    ns.forward, ns.mcmc, ns.measurements, ns.prior, ns.sht, ns.transforms, ns.utils = (
        forward, mcmc, measurements, prior, sht, transforms, utils)
    return ns


# ------------------------------------------------------------------ elementwise
def test_soft_known_answers_bit_exact(px):
    # reference tests/test_utils.py:35-44 (exact ==)
    soft = px.utils.soft
    assert all(soft([1, 2, 3], T=2) == [0, 0, 1])
    assert all(soft([-1, -2, -3], T=2) == [0, 0, -1])
    assert all(soft([1 + 1j, 0.5 - 0.5j, 0], T=1) == [(1 + 1j) * (np.sqrt(2) - 1) / np.sqrt(2), 0, 0])


def test_soft_golden_bit_exact(px):
    g = golden("ref_soft.npz")
    soft = px.utils.soft
    assert np.array_equal(soft(g["xr"], 0.8), g["soft_r_scalar"])
    assert np.array_equal(soft(g["xr"], g["tv"]), g["soft_r_vec"])
    assert np.array_equal(soft(g["xc"], 1.0), g["soft_c_scalar"])
    assert np.array_equal(soft(g["xc"], g["tv"]), g["soft_c_vec"])


def test_soft_edge_cases(px):
    soft = px.utils.soft
    assert soft(np.zeros(0), 1.0).size == 0                       # empty
    x = np.array([0.0, -0.0, 1e-300, -1e300, 0.25, -0.25])
    assert np.array_equal(soft(x, 0.25), [0, 0, 0, -1e300 + 0.25, 0, 0])  # |x| == T zeroed (inclusive)
    big = np.random.default_rng(1).standard_normal(1 << 20)       # larger than one grid pass
    from oracle import pxmcmc_ref as R
    assert np.array_equal(soft(big, 0.5), R.soft(big, 0.5))


def test_l1_prox_matches_soft(px):
    # reference tests/test_proxes.py:17-21
    X = np.arange(100)
    for setting in ("synthesis",):
        reg = px.prior.L1(setting, lambda v: v, lambda v: v, 50)
        assert np.all(reg.proxf(X) == px.utils.soft(X, 50))
    reg = px.prior.L1("analysis", lambda v: v, lambda v: v, 50)
    assert np.allclose(reg.proxf(X), px.utils.soft(X, 50))


# ------------------------------------------------------------------ SHT primitives
@pytest.mark.parametrize("spin", [0, 2])
def test_sht_golden(px, spin):
    g = golden("ref_sht_L12.npz")
    L = int(g["L"])
    s = px.sht
    assert rel_l2(s.inverse(g[f"flm_s{spin}"], L, Spin=spin), g[f"inverse_s{spin}"]) < TOL
    assert rel_l2(s.forward(g["f"], L, Spin=spin), g[f"forward_s{spin}"]) < TOL
    assert rel_l2(s.inverse_adjoint(g["f"], L, Spin=spin), g[f"inverse_adjoint_s{spin}"]) < TOL
    assert rel_l2(s.forward_adjoint(g[f"flm_s{spin}"], L, Spin=spin), g[f"forward_adjoint_s{spin}"]) < TOL


@pytest.mark.parametrize("L,spin", [(3, 0), (4, 2), (17, 0), (33, 2), (64, 0), (100, -2)])
def test_sht_vs_oracle_and_properties(px, L, spin):
    from oracle import ssht_ref

    rng = np.random.default_rng(100 + L)
    s = px.sht
    flm = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    flm[: spin * spin] = 0
    f = rng.standard_normal((L, 2 * L - 1)) + 1j * rng.standard_normal((L, 2 * L - 1))
    fi = s.inverse(flm, L, Spin=spin)
    assert rel_l2(fi, ssht_ref.inverse(flm, L, spin)) < TOL
    assert rel_l2(s.forward(f, L, Spin=spin), ssht_ref.forward(f, L, spin)) < TOL
    assert rel_l2(s.inverse_adjoint(f, L, Spin=spin), ssht_ref.inverse_adjoint(f, L, spin)) < TOL
    assert rel_l2(s.forward_adjoint(flm, L, Spin=spin), ssht_ref.forward_adjoint(flm, L, spin)) < TOL
    # exactness and adjointness (reference tests/test_measurements.py, test_utils.py:85-100)
    assert rel_l2(s.forward(fi, L, Spin=spin), flm) < TOL
    assert abs(np.vdot(f, fi) - np.vdot(s.inverse_adjoint(f, L, Spin=spin), flm)) < 1e-9 * np.linalg.norm(f) * np.linalg.norm(fi)


def test_sht_batched_equals_single(px):
    import torch
    from pxmcmc_b200 import device as D

    L, nb = 20, 7
    rng = np.random.default_rng(5)
    flm = rng.standard_normal((nb, L * L)) + 1j * rng.standard_normal((nb, L * L))
    out = D.to_host(D.ShtPlan.get(L, 0, nb).inverse(D.to_dev_c(flm)))
    for i in range(nb):
        assert rel_l2(out[i], px.sht.inverse(flm[i], L).ravel()) < 1e-13
    back = D.to_host(D.ShtPlan.get(L, 0, nb).forward(D.to_dev_c(out)))
    assert rel_l2(back, flm) < TOL


def test_sht_large_bandlimit_properties(px):
    """size-independent properties at the BASELINE bandlimit: exact round trip and linearity"""
    L = 256
    rng = np.random.default_rng(9)
    flm = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    f = px.sht.inverse(flm, L)
    assert rel_l2(px.sht.forward(f, L), flm) < TOL
    g = rng.standard_normal(f.shape) + 1j * rng.standard_normal(f.shape)
    a = px.sht.inverse_adjoint(g, L)
    assert abs(np.vdot(g, f) - np.vdot(a, flm)) < 1e-10 * np.linalg.norm(g) * np.linalg.norm(f)


# ------------------------------------------------------------------ wavelets
@pytest.mark.parametrize("tag", ["L10B2", "L16B1p5"])
def test_wavelet_golden(px, tag):
    g = golden(f"ref_wavelet_{tag}.npz")
    L, B, J = int(g["L"]), float(g["B"]), int(g["J_min"])
    t = px.transforms.SphericalWaveletTransform(L, B, J)
    assert (t.nscal, t.nwav, t.ncoefs) == (int(g["nscal"]), int(g["nwav"]), int(g["nscal"]) + int(g["nwav"]))
    assert rel_l2(t.forward(g["x_pix"]), g["forward"]) < TOL
    assert rel_l2(t.inverse(g["x_coef"]), g["inverse"]) < TOL
    assert rel_l2(t.inverse_adjoint(g["x_pix"]), g["inverse_adjoint"]) < TOL
    assert rel_l2(t.forward_adjoint(g["x_coef"]), g["forward_adjoint"]) < TOL
    # prior weight vectors of the S2 priors
    assert rel_l2(px.prior.S2_Wavelets_L1("synthesis", None, None, 1.0, L, B, J).T, g["s2_T"]) < 1e-14
    pw = px.prior.S2_Wavelets_L1_Power_Weights("synthesis", None, None, 1.0, L, B, J, eta=1)
    assert rel_l2(pw.T, g["s2pw_T"]) < 1e-14 and rel_l2(pw.map_weights, g["s2pw_w"]) < 1e-14


@pytest.mark.parametrize("L,B,J", [(10, 2, 2), (32, 1.5, 2), (28, 2, 2), (64, 3, 1)])
def test_wavelet_vs_oracle_and_reference_properties(px, L, B, J):
    from oracle import pxmcmc_ref as R

    rng = np.random.default_rng(L)
    t = px.transforms.SphericalWaveletTransform(L, B, J)
    o = R.WaveletTransform(L, B, J)
    assert t.ncoefs == o.ncoefs and t.nscal == o.nscal
    xp = rng.standard_normal(L * (2 * L - 1)) + 1j * rng.standard_normal(L * (2 * L - 1))
    xc = rng.standard_normal(t.ncoefs) + 1j * rng.standard_normal(t.ncoefs)
    assert rel_l2(t.inverse(xc), o.inverse(xc)) < TOL
    assert rel_l2(t.inverse_adjoint(xp), o.inverse_adjoint(xp)) < TOL
    assert rel_l2(t.forward(xp), o.forward(xp)) < TOL
    assert rel_l2(t.forward_adjoint(xc), o.forward_adjoint(xc)) < TOL
    # reference tests/test_transforms.py:16-46 on a band-limited real map
    x = px.sht.inverse(px.sht.forward(xp.real, L), L).ravel()
    assert np.allclose(t.inverse(t.forward(x)), x)
    assert np.isclose(np.vdot(xc, t.forward(x)) - np.vdot(t.forward_adjoint(xc), x), 0, atol=1e-8)
    assert np.isclose(np.vdot(x, t.inverse(xc)) - np.vdot(t.inverse_adjoint(x), xc), 0, atol=1e-8)


def test_wavelet_full_size_properties(px):
    """BASELINE size (L=256, B=1.5): dot test of the hot pair and exact reconstruction"""
    L, B, J = 256, 1.5, 2
    rng = np.random.default_rng(3)
    t = px.transforms.SphericalWaveletTransform(L, B, J)
    assert t.ncoefs == 398342
    xc = rng.standard_normal(t.ncoefs) + 1j * rng.standard_normal(t.ncoefs)
    xp = rng.standard_normal(L * (2 * L - 1)) + 1j * rng.standard_normal(L * (2 * L - 1))
    y, g = t.inverse(xc), t.inverse_adjoint(xp)
    assert abs(np.vdot(xp, y) - np.vdot(g, xc)) < 1e-10 * np.linalg.norm(xp) * np.linalg.norm(y)
    x = px.sht.inverse(px.sht.forward(xp, L), L).ravel()
    assert rel_l2(t.inverse(t.forward(x)), x) < TOL


# ------------------------------------------------------------------ operators
def test_operator_output_lengths(px):
    # reference tests/test_forward.py
    L, B, J = 10, 2, 2
    rng = np.random.default_rng(0)
    data = rng.standard_normal(L * (2 * L - 1))
    for setting in ("analysis", "synthesis"):
        for sig in (0.1, np.full(data.size, 0.1)):
            op = px.forward.SphericalWaveletTransformOperator(data, sig, setting, L, B, J)
            assert len(op.forward(rng.random(op.nparams).astype(complex))) == len(op.data)
            assert len(op.calc_gradg(rng.random(len(op.data)))) == op.nparams
            A = sparse.random(len(data), L * (2 * L - 1), density=0.05, random_state=1)
            op = px.forward.PathIntegralOperator(A, data, sig, setting, L, B, J)
            assert len(op.forward(rng.random(op.nparams).astype(complex))) == len(op.data)
            assert len(op.calc_gradg(rng.random(len(op.data)))) == op.nparams
    with pytest.raises(ValueError):
        px.forward.ForwardOperator(data, 0.1, "nonsense")
    with pytest.raises(TypeError):
        px.forward.ForwardOperator(data, np.ones(3), "analysis")


def test_pathintegral(px):
    # reference tests/test_measurements.py:8-45
    L = 10
    rng = np.random.default_rng(2)
    A = sparse.random(100, L * (2 * L - 1), density=0.05, random_state=2, format="csr")
    p = px.measurements.PathIntegral(A)
    x = rng.standard_normal(L * (2 * L - 1)) + 1j * rng.standard_normal(L * (2 * L - 1))
    y = rng.random(100) + 0j
    assert rel_l2(p.forward(x), A @ x) < 1e-14
    assert rel_l2(p.adjoint(y), A.T @ y) < 1e-14
    ring = np.zeros((L, 2 * L - 1))
    ring[(L - 1) // 2, :] = 2 * np.pi / (2 * L - 1)
    pr = px.measurements.PathIntegral(sparse.csr_matrix(ring.reshape(1, -1)))
    assert np.isclose(pr.forward(np.ones(L * (2 * L - 1)))[0], 2 * np.pi)
    empty = px.measurements.PathIntegral(sparse.csr_matrix((5, L * (2 * L - 1))))   # rows without entries
    assert np.all(empty.forward(x) == 0)
    # a batch of chains reads the matrix once per group of four chains: ragged batch sizes, both directions
    from pxmcmc_b200 import device as D

    for nb in (2, 4, 7):
        xb = rng.standard_normal((nb, L * (2 * L - 1))) + 1j * rng.standard_normal((nb, L * (2 * L - 1)))
        yb = rng.standard_normal((nb, 100)) + 1j * rng.standard_normal((nb, 100))
        fb = p.forward(D.to_dev_c(xb)).cpu().numpy()
        ab = p.adjoint(D.to_dev_c(yb)).cpu().numpy()
        for c in range(nb):
            assert np.array_equal(fb[c], p.forward(xb[c])) and np.array_equal(ab[c], p.adjoint(yb[c]))


def test_weaklensing_golden(px):
    g = golden("ref_weaklensing_L12.npz")
    L = int(g["L"])
    wl = px.measurements.WeakLensing(L, mask=g["mask"], ngal=g["ngal"])
    assert np.array_equal(wl.harmonic_kernel, g["kernel"])
    assert rel_l2(wl.inv_cov, g["inv_cov"]) < 1e-15
    assert rel_l2(wl.forward(g["kappa"]), g["forward"]) < TOL
    assert rel_l2(wl.adjoint(g["gamma"]), g["adjoint"]) < TOL
    wl0 = px.measurements.WeakLensing(L)
    assert rel_l2(wl0.forward(g["kappa"]), g["forward_nomask"]) < TOL
    assert rel_l2(wl0.adjoint(g["kappa"]), g["adjoint_nomask"]) < TOL
    a = abs(np.vdot(g["kappa"], wl.adjoint(g["gamma"])))
    b = abs(np.vdot(g["gamma"], wl.forward(g["kappa"])))
    assert np.isclose(a, b)
    t = px.transforms.SphericalWaveletTransform(L, 2, 2)
    fo = px.forward.ForwardOperator(g["gdata"], 1 / wl.inv_cov, "synthesis", transform=t, measurement=wl, nparams=t.ncoefs)
    assert rel_l2(fo.invcov.diagonal(), g["op_invcov"]) < 1e-15
    # default: harmonic-space composition (the two cancelling full-L SHTs of each direction skipped, SURVEY 3.5) ...
    assert fo._fused()
    assert rel_l2(fo.forward(g["X"]), g["op_forward"]) < TOL
    assert rel_l2(fo.calc_gradg(g["op_forward"]), g["op_gradg"]) < TOL
    # ... and the reference's literal composition through pixel space
    fo.fuse_harmonic = False
    assert not fo._fused()

    class Doubled(px.measurements.WeakLensing):  # a user subclass that overrides forward must not be bypassed
        def forward(self, kappa):
            return 2 * super().forward(kappa)

    fo2 = px.forward.ForwardOperator(g["gdata"], 1 / wl.inv_cov, "synthesis", transform=t, nparams=t.ncoefs,
                                     measurement=Doubled(L, mask=g["mask"], ngal=g["ngal"]))
    assert not fo2._fused() and rel_l2(fo2.forward(g["X"]), 2 * g["op_forward"]) < TOL
    assert rel_l2(fo.forward(g["X"]), g["op_forward"]) < TOL
    assert rel_l2(fo.calc_gradg(g["op_forward"]), g["op_gradg"]) < TOL
    with pytest.raises(ValueError):
        px.measurements.WeakLensing(L, mask=np.ones((3, 3)))
    with pytest.raises(ValueError):
        px.measurements.WeakLensing(0)


# ------------------------------------------------------------------ samplers
def _myula_from_golden(px, g, **kw):
    L, B, J = int(g["L"]), float(g["B"]), int(g["J_min"])
    sig = g["sig_d"] if g["sig_d"].ndim else float(g["sig_d"])
    op = px.forward.SphericalWaveletTransformOperator(g["data"], sig, "synthesis", L, B, J)
    p = px.mcmc.PxMCMCParams(nsamples=int(g["nsamples"]), nburn=int(g["nburn"]), ngap=int(g["ngap"]),
                             delta=float(g["delta"]), lmda=float(g["lmda"]), mu=float(g["mu"]), verbosity=0,
                             track=["logposterior", "L2", "prior", "chain", "predictions"])
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu, L=L, B=B, J_min=J)
    return px.mcmc.MYULA(op, reg, p, **kw)


@pytest.mark.parametrize("tag", ["L10_complex", "L10_real_sigvec", "L16B1p5_complex"])
def test_myula_chain_reproduces_reference(px, tag):
    """seeded run with host noise == the unmodified reference's chain"""
    import warnings

    g = golden(f"ref_myula_{tag}.npz")
    m = _myula_from_golden(px, g)
    np.random.seed(int(g["seed"]))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.run()
    assert rel_l2(m.chain, g["chain"]) < TOL
    assert rel_l2(m.preds, g["preds"]) < TOL
    assert rel_l2(m.logPi, g["logPi"]) < TOL
    assert rel_l2(m.L2s, g["L2s"]) < TOL
    assert rel_l2(m.priors, g["priors"]) < TOL


def test_myula_single_step_golden(px):
    g = golden("ref_myula_step_L10.npz")
    L, B, J = int(g["L"]), float(g["B"]), int(g["J_min"])
    op = px.forward.SphericalWaveletTransformOperator(g["data"], float(g["sig_d"]), "synthesis", L, B, J)
    p = px.mcmc.PxMCMCParams(delta=float(g["delta"]), lmda=float(g["lmda"]), mu=float(g["mu"]), verbosity=0, nsamples=1)
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu, L=L, B=B, J_min=J)
    m = px.mcmc.MYULA(op, reg, p)
    assert rel_l2(op.invcov.diagonal(), g["invcov"]) < 1e-15
    assert rel_l2(reg.T, g["T"]) < 1e-14
    assert rel_l2(op.forward(g["X"]), g["preds"]) < TOL
    assert rel_l2(op.calc_gradg(g["preds"]), g["gradg"]) < TOL
    prox = reg.proxf(g["X"])
    assert np.array_equal(prox == 0, g["prox"] == 0)                      # support identical
    assert np.array_equal(np.sign(prox.real), np.sign(g["prox"].real))    # sign pattern identical
    assert np.array_equal(np.sign(prox.imag), np.sign(g["prox"].imag))
    assert rel_l2(prox, g["prox"]) < 1e-15
    np.random.seed(5)
    assert rel_l2(m.chain_step(g["X"], g["prox"], g["gradg"]), g["Xn"]) < 1e-14
    lp, l2, pr = m.logpi(g["X"], g["preds"])
    assert np.isclose(lp, g["logpi"], rtol=1e-11) and np.isclose(l2, g["L2"], rtol=1e-11) and np.isclose(pr, g["prior"], rtol=1e-12)


def test_pxmala_reproduces_reference(px):
    import warnings

    g = golden("ref_pxmala_L10.npz")
    L, B, J = int(g["L"]), float(g["B"]), int(g["J_min"])
    op = px.forward.SphericalWaveletTransformOperator(g["data"], float(g["sig_d"]), "analysis", L, B, J)
    p = px.mcmc.PxMCMCParams(nsamples=int(g["nsamples"]), nburn=int(g["nburn"]), ngap=int(g["ngap"]),
                             delta=float(g["delta"]), lmda=float(g["lmda"]), mu=float(g["mu"]), verbosity=0,
                             track=["logposterior", "L2", "prior", "chain", "predictions"])
    reg = px.prior.L1("analysis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu)
    m = px.mcmc.PxMALA(op, reg, p, tune_delta=True)
    assert np.isclose(m.calc_logtransition(g["X1"], g["X2"], g["proxf"], g["gradg"]), g["logtrans"], rtol=1e-10)
    assert rel_l2(reg.proxf(g["X1"]), g["proxf"]) < TOL
    np.random.seed(int(g["seed"]))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.run()
    assert list(m.acceptance_trace) == list(g["acceptance_trace"])
    assert np.allclose(m.deltas_trace, g["deltas_trace"], rtol=1e-13, atol=0)
    assert rel_l2(m.chain, g["chain"]) < TOL
    assert rel_l2(m.logPi, g["logPi"]) < TOL


def test_skrock_reproduces_reference(px):
    g = golden("ref_skrock_L10.npz")
    L, B, J = int(g["L"]), float(g["B"]), int(g["J_min"])
    A = sparse.csr_matrix((g["A_data"], g["A_indices"], g["A_indptr"]), shape=tuple(g["A_shape"]))
    op = px.forward.PathIntegralOperator(A, g["data"], g["sig_d"], "synthesis", L, B, J)
    p = px.mcmc.PxMCMCParams(delta=float(g["delta"]), lmda=float(g["lmda"]), mu=float(g["mu"]), s=3, verbosity=0, nsamples=1)
    reg = px.prior.S2_Wavelets_L1_Power_Weights("synthesis", op.transform.inverse, op.transform.inverse_adjoint,
                                               p.lmda * p.mu, L=L, B=B, J_min=J, eta=1)
    m = px.mcmc.SKROCK(op, reg, p)
    assert np.allclose(m.mus, g["mus"], rtol=1e-13) and np.allclose(m.nus, g["nus"], rtol=1e-13) and np.allclose(m.ks, g["ks"], rtol=1e-13)
    m5 = px.mcmc.SKROCK(op, reg, px.mcmc.PxMCMCParams(s=5, verbosity=0, nsamples=1))
    assert np.allclose(m5.mus, g["mus5"], rtol=1e-13) and np.allclose(m5.nus, g["nus5"], rtol=1e-13)
    assert rel_l2(reg.T, g["T"]) < 1e-14
    assert np.isclose(reg.prior(g["X"]), g["prior"], rtol=1e-12)
    assert rel_l2(op.forward(g["X"]), g["preds"]) < TOL
    assert rel_l2(op.calc_gradg(g["preds"]), g["gradg"]) < TOL
    assert rel_l2(m._gradlogpi(g["X"]), g["gradlogpi"]) < TOL
    np.random.seed(31)
    assert rel_l2(m.chain_step(g["X"]), g["Xn"]) < TOL


def test_samplers_smoke_identity_operators(px):
    """reference tests/test_mcmc.py: each sampler runs with IdentityTransform + Identity + L1"""
    rng = np.random.default_rng(0)
    data = rng.standard_normal(190)
    for setting in ("analysis", "synthesis"):
        for sig in (0.1, np.full(190, 0.1)):
            t = px.transforms.IdentityTransform()
            op = px.forward.ForwardOperator(data, sig, setting, t, px.measurements.Identity(190, 190), nparams=190)
            reg = px.prior.L1(setting, t.inverse, t.inverse_adjoint, 1)
            prm = px.mcmc.PxMCMCParams(nsamples=20, nburn=5, ngap=2, verbosity=0, s=5)
            for cls in (px.mcmc.MYULA, px.mcmc.PxMALA, px.mcmc.SKROCK):
                algo = cls(op, reg, prm)
                algo.run()
                algo = cls(op, reg, prm)
                algo.run(data.copy())
                with pytest.raises(Exception):
                    cls(op, reg, prm).run(data[:5])
                with pytest.raises(TypeError):
                    cls(op, reg, prm).run([1.0] * 190)


def test_multichain_device_noise(px):
    """batched chains with Philox noise: chains differ, statistics sane, batch == plan batch"""
    L, B, J, nb = 16, 2, 2, 4
    rng = np.random.default_rng(4)
    data = px.sht.inverse(rng.standard_normal(L * L) + 0j, L).ravel()
    op = px.forward.SphericalWaveletTransformOperator(data, 0.1, "synthesis", L, B, J, nchains=nb)
    p = px.mcmc.PxMCMCParams(nsamples=3, nburn=0, ngap=2, delta=1e-6, lmda=1e-6, verbosity=0)
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda, L=L, B=B, J_min=J)
    m = px.mcmc.MYULA(op, reg, p, noise="device", nchains=nb, seed=7)
    m.run(np.zeros(op.nparams))
    assert m.chain.shape == (nb, 3, op.nparams)
    assert np.all(np.isfinite(m.chain))
    assert not np.allclose(m.chain[0], m.chain[1])
    # identical seed => identical chains (counter-based generator)
    m2 = px.mcmc.MYULA(op, reg, p, noise="device", nchains=nb, seed=7)
    m2.run(np.zeros(op.nparams))
    assert np.array_equal(m.chain, m2.chain)
    # run() replays the iteration as a CUDA graph when the noise is generated on the device: same chain as the eager loop
    m3 = px.mcmc.MYULA(op, reg, p, noise="device", nchains=nb, seed=7)
    m3.graph_run = False
    m3.run(np.zeros(op.nparams))
    assert np.array_equal(m.chain, m3.chain) and np.array_equal(m.logPi, m3.logPi)
    # first increment is sqrt(2 delta) * N(0,1) to leading order
    z = m.chain[:, 0, :].ravel() / np.sqrt(2e-6)
    assert abs(z.std() - np.sqrt(1.0)) < 0.2


# ------------------------------------------------------------------ HEALPix (SURVEY.md 8 a13)
@pytest.mark.parametrize("nside,L", [(8, 12), (16, 40), (4, 3)])
def test_healpix_against_oracle(px, nside, L):
    """utils.alm2map / utils.map2alm (healpy's, as the reference wraps them) against the dense-Y_lm oracle"""
    from oracle import healpix_ref as H

    rng = np.random.default_rng(2)
    Y = H.ylm_matrix(nside, L)
    alm = np.zeros(H.alm_size(L - 1), complex)
    for el in range(L):
        for m in range(el + 1):
            alm[H.alm_index(el, m, L - 1)] = rng.standard_normal() + (1j * rng.standard_normal() if m else 0)
    mp = px.utils.alm2map(alm, nside)
    assert mp.dtype == np.float64 and mp.shape == (12 * nside * nside,)
    assert rel_l2(mp, H.alm2map(alm, nside, Y)) < TOL
    noisy = mp + rng.standard_normal(mp.size)  # not band-limited: the iterations matter
    for it in (0, 3):
        assert rel_l2(px.utils.map2alm(noisy, L - 1, iter=it), H.map2alm(noisy, L - 1, iter=it, Y=Y)) < TOL
    assert rel_l2(px.utils.map2alm(noisy, L - 1), H.map2alm(noisy, L - 1, iter=3, Y=Y)) < TOL  # healpy default
    # the reference's HEALPix -> MW data path (experiments/earthtopography/main.py:80-82)
    from oracle import ssht_ref

    flm = px.utils.lm_hp2lm(px.utils.map2alm(noisy, L - 1), L)
    mw = px.utils.alm2map_mw(flm, L, 0)
    assert rel_l2(mw, ssht_ref.inverse(H.lm_hp2lm(H.map2alm(noisy, L - 1, Y=Y), L), L, 0).ravel()) < TOL


def test_healpix_full_size_properties(px):
    """nside 256, lmax 255 (the reference's ETOPO1 preparation): spot values against scipy's Y_lm,
    Euclidean adjointness of the two device transforms, monopole, round trip"""
    import torch
    from scipy.special import sph_harm_y

    from oracle import healpix_ref as H
    from pxmcmc_b200 import device as D

    nside, L = 256, 256
    npix = 12 * nside * nside
    rng = np.random.default_rng(4)
    plan = px.utils._HealpixPlan.get(nside, L)
    x = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    g = rng.standard_normal(npix) + 1j * rng.standard_normal(npix)
    fx = D.to_host(plan.synth(D.to_dev_c(x)))
    ag = D.to_host(plan.adjoint(D.to_dev_c(g)))
    lhs, rhs = np.vdot(g, fx), np.vdot(ag, x)
    assert abs(lhs - rhs) < 1e-11 * abs(lhs)
    theta, phi = H.pix2ang(nside)
    els = np.concatenate([np.full(2 * el + 1, el) for el in range(L)])
    ms = np.concatenate([np.arange(-el, el + 1) for el in range(L)])
    for p in (0, 3, 7, 1234, npix // 2 + 17, npix - 1, 2 * nside * (nside - 1) + 5):
        exact = np.sum(x * sph_harm_y(els, ms, theta[p], phi[p]))
        assert abs(fx[p] - exact) < 1e-10 * np.abs(fx).max()
    a00 = px.utils.map2alm(np.full(npix, -3.0), L - 1, iter=0)[0]
    assert np.isclose(a00, -3.0 * np.sqrt(4 * np.pi), rtol=1e-12)
    alm = px.utils.lm2lm_hp(px.utils.lm_hp2lm(H.lm2lm_hp(x, L) * (np.arange(H.alm_size(L - 1)) >= 0), L), L)
    alm[:L] = alm[:L].real  # m = 0 coefficients of a real map are real
    back = px.utils.map2alm(px.utils.alm2map(alm, nside), L - 1)
    assert rel_l2(back, alm) < 1e-5  # HEALPix quadrature + 3 refinements (not exact, as in healpy)
    torch.cuda.synchronize()


# ------------------------------------------------------------------ CUDA-graph replay of the iteration
@pytest.mark.parametrize("iters_per_graph", [1, 3])
def test_myula_graph_replay_matches_eager(px, iters_per_graph):
    """a captured MYULA iteration (one launch) follows exactly the eager chain: same kernels, same
    Philox stream (the step counter lives on the device and advances inside the graph)"""
    import torch

    from pxmcmc_b200 import device as D

    L, B, J = 24, 2.0, 1
    rng = np.random.default_rng(8)
    data = rng.standard_normal(L * (2 * L - 1)) + 0j
    prm = px.mcmc.PxMCMCParams(delta=1e-4, lmda=2e-4, mu=1.0, nsamples=1, verbosity=0, track=[])

    def make():
        op = px.forward.SphericalWaveletTransformOperator(data, 0.7, "synthesis", L, B, J)
        reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 3e-3, L=L, B=B, J_min=J)
        return op, px.mcmc.MYULA(op, reg, prm, noise="device", seed=77, stream0=5)

    op, eager = make()
    X0 = D.to_dev_c(rng.laplace(size=(1, op.nparams)))
    P0 = eager._initial_preds(X0)  # the form run() carries the predictions in (ring coefficients for this operator)
    X, P = X0, P0
    for _ in range(6):
        X, P = eager.iterate(X, P)
    _, graphed = make()
    chain = graphed.capture(X0, P0, iterations=iters_per_graph)
    for _ in range(6 // iters_per_graph):
        chain.step()
    torch.cuda.synchronize()
    Xg, Pg = chain.state()
    assert torch.equal(Xg, X) and torch.equal(Pg, eager._pix(P))  # bit-identical
    assert graphed._step_counter == eager._step_counter == 6
    # an eager call after the capture draws the host counter, which the replays advanced
    assert graphed._dstep is None
    Xg, _ = graphed.iterate(*chain._state_raw())
    X, P = eager.iterate(X, P)
    assert torch.equal(Xg, X) and graphed._step_counter == eager._step_counter == 7
    with pytest.raises(ValueError):
        px.mcmc.MYULA(op, eager.prior, prm, noise="host").capture(X0, eager._pix(P0))


@pytest.mark.parametrize("mode,nb", [(2, 2), (3, 2), (3, 3), (3, 9)])
def test_ring_fft_two_pass_against_multipass(px, mode, nb):
    """the two-pass ring FFT (mode 2: all Bluestein lengths <= 1024; mode 3: its persistent, TMA-staged
    variant for lengths 512 / 1024, with even and odd item counts; the development builds -DPXM_FFT_PAIRSPLIT / _PINGPONG
    add modes 5 / 4 for their kernels) against the
    independent multi-pass kernel (the path lengths > 1024 take), through all four wavelet operators at the
    BASELINE bandlimit"""
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D

    L, B, J = 256, 1.5, 2
    rng = np.random.default_rng(13)
    plan = D.WaveletPlan.get(L, B, J, nb)
    coef = D.to_dev_c(rng.standard_normal((nb, plan.ncoefs)) + 1j * rng.standard_normal((nb, plan.ncoefs)))
    pix = D.to_dev_c(rng.standard_normal((nb, plan.npix)) + 1j * rng.standard_normal((nb, plan.npix)))
    for name, x in (("synthesis", coef), ("synthesis_adjoint", pix), ("analysis", pix), ("analysis_adjoint", coef)):
        try:
            _lib.check(_lib.lib.pxm_debug_set_fft_multipass(mode))
            fast = D.to_host(getattr(plan, name)(x))
            _lib.check(_lib.lib.pxm_debug_set_fft_multipass(1))
            slow = D.to_host(getattr(plan, name)(x))
        finally:
            _lib.check(_lib.lib.pxm_debug_set_fft_multipass(0))
        assert rel_l2(fast, slow) < 1e-13, name


def test_iterate_host_pipeline_matches_device_iteration(px):
    """the pipelined host-buffer iteration (chain groups on three streams) gives exactly the batch
    iteration: same chains, same Philox streams, whatever the grouping"""
    import torch

    from pxmcmc_b200 import device as D

    L, B, J, nch = 16, 2.0, 1, 16
    rng = np.random.default_rng(5)
    data = rng.standard_normal(L * (2 * L - 1)) + 0j
    prm = px.mcmc.PxMCMCParams(delta=1e-4, lmda=2e-4, mu=1.0, nsamples=1, verbosity=0, track=[])
    op = px.forward.SphericalWaveletTransformOperator(data, 0.7, "synthesis", L, B, J, nchains=nch)
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 3e-3, L=L, B=B, J_min=J)
    X0 = rng.laplace(size=(nch, op.nparams)) + 0j
    P0 = D.to_host(op.forward(D.to_dev_c(X0)))
    ref = px.mcmc.MYULA(op, reg, prm, noise="device", nchains=nch, seed=9, stream0=3)
    Xr, Pr = ref.iterate(D.to_dev_c(X0), D.to_dev_c(P0))
    for groups in (1, 4, [1, 3, 4, 8]):
        m = px.mcmc.MYULA(op, reg, prm, noise="device", nchains=nch, seed=9, stream0=3)
        Xh, Ph = torch.from_numpy(X0.copy()).pin_memory(), torch.from_numpy(P0.copy()).pin_memory()
        Xo, Po = torch.empty_like(Xh).pin_memory(), torch.empty_like(Ph).pin_memory()
        m.iterate_host(Xh, Ph, Xo, Po, groups=groups)
        assert torch.equal(Xo, Xr.cpu()) and torch.equal(Po, Pr.cpu()), groups
        assert m._step_counter == 1


@pytest.mark.parametrize("mode", [2, 3])
def test_ring_fft_two_pass_all_radices_against_oracle(px, mode):
    """two-pass ring FFT forced on (mode 2; mode 3: persistent staged kernel for length 512, ragged
    item count) at L=70, B=2: Bluestein lengths 16...512, i.e. every radix pair below (32, 32), paired
    (spin 0) and unpaired (spin 2) ring layouts, against the CPU oracle"""
    from oracle import pxmcmc_ref as R
    from oracle import ssht_ref
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D

    L, B, J = 70, 2.0, 2
    rng = np.random.default_rng(17)
    t = R.WaveletTransform(L, B, J)
    plan = D.WaveletPlan.get(L, B, J, 3)
    assert sorted(set(plan.bandlimits)) == [4, 8, 16, 32, 64, 70]
    coef = rng.standard_normal((3, plan.ncoefs)) + 1j * rng.standard_normal((3, plan.ncoefs))
    pix = rng.standard_normal((3, plan.npix)) + 1j * rng.standard_normal((3, plan.npix))
    flm = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    flm[:4] = 0
    try:
        _lib.check(_lib.lib.pxm_debug_set_fft_multipass(mode))
        got = {"synthesis": D.to_host(plan.synthesis(D.to_dev_c(coef))), "synthesis_adjoint": D.to_host(plan.synthesis_adjoint(D.to_dev_c(pix))),
               "analysis": D.to_host(plan.analysis(D.to_dev_c(pix))), "analysis_adjoint": D.to_host(plan.analysis_adjoint(D.to_dev_c(coef)))}
        s2 = D.ShtPlan.get(L, 2, 1)
        got_s2 = {"inverse": D.to_host(s2.inverse(D.to_dev_c(flm))), "forward": D.to_host(s2.forward(D.to_dev_c(pix[0]))),
                  "inverse_adjoint": D.to_host(s2.inverse_adjoint(D.to_dev_c(pix[0]))), "forward_adjoint": D.to_host(s2.forward_adjoint(D.to_dev_c(flm)))}
    finally:
        _lib.check(_lib.lib.pxm_debug_set_fft_multipass(0))
    for c in range(3):
        assert rel_l2(got["synthesis"][c], t.inverse(coef[c])) < TOL
        assert rel_l2(got["synthesis_adjoint"][c], t.inverse_adjoint(pix[c])) < TOL
        assert rel_l2(got["analysis"][c], t.forward(pix[c])) < TOL
        assert rel_l2(got["analysis_adjoint"][c], t.forward_adjoint(coef[c])) < TOL
    assert rel_l2(got_s2["inverse"], ssht_ref.inverse(flm, L, 2).ravel()) < TOL
    assert rel_l2(got_s2["forward"], ssht_ref.forward(pix[0].reshape(L, 2 * L - 1), L, 2)) < TOL
    assert rel_l2(got_s2["inverse_adjoint"], ssht_ref.inverse_adjoint(pix[0].reshape(L, 2 * L - 1), L, 2)) < TOL
    assert rel_l2(got_s2["forward_adjoint"], ssht_ref.forward_adjoint(flm, L, 2).ravel()) < TOL


@pytest.mark.parametrize("L", [512, 1024])
def test_large_bandlimit_adjointness_and_exactness(px, L):
    """the upper end of the north-star range (L <= 1024; Bluestein lengths 2048 / 4096 -> multi-pass ring FFT,
    23 GiB of Legendre tables at L = 1024): Euclidean dot-tests of both operator pairs and the exactness of
    synthesis(analysis(f)) on a band-limited f, the properties the reference's tests/test_transforms.py:16-46
    assert at L = 10"""
    import torch

    from pxmcmc_b200 import device as D

    plan = D.WaveletPlan(L, 2.0, 2, 1)  # not cached: the tables are released with the plan
    g = torch.Generator(device="cuda").manual_seed(3)

    def rnd(n):
        return torch.randn(n, dtype=torch.float64, device="cuda", generator=g) + 1j * torch.randn(n, dtype=torch.float64, device="cuda", generator=g)

    x, y = rnd(plan.ncoefs), rnd(plan.npix)
    syn, syn_adj, ana, ana_adj = plan.synthesis(x), plan.synthesis_adjoint(y), plan.analysis(y), plan.analysis_adjoint(x)
    d1, d2 = torch.vdot(y, syn), torch.vdot(x, ana)
    assert abs(d1 - torch.vdot(syn_adj, x)) / abs(d1) < TOL
    assert abs(d2 - torch.vdot(ana_adj, y)) / abs(d2) < TOL
    back = plan.synthesis(plan.analysis(syn))
    assert float((back - syn).abs().pow(2).sum().sqrt() / syn.abs().pow(2).sum().sqrt()) < TOL
    from pxmcmc_b200._lib import check, lib

    check(lib.pxm_wav_plan_destroy(plan.h))
    plan.h = None


def test_credible_interval_ranges_match_the_reference_bit_for_bit(px):
    """pxmcmc/uncertainty.py through the GPU column-quantile kernel against the vectors the unmodified
    reference produced (np.quantile, method "linear"): ragged column counts, 37 to 5000 samples
    (padded to the next power of two in shared memory), ties; == not allclose"""
    import torch

    from oracle.gen_golden_uncertainty import CASES, make_chain
    from pxmcmc_b200 import uncertainty as U

    g = golden("ref_uncertainty.npz")
    for i, (n, p, seed) in enumerate(CASES):
        chain = make_chain(n, p, seed)
        assert np.array_equal(U.credible_interval_range(chain), g[f"ci_{i}"])
        assert np.array_equal(U.credible_interval_range(chain, alpha=0.1), g[f"ci10_{i}"])
        dev = U.credible_interval_range(torch.from_numpy(chain).cuda())
        assert isinstance(dev, torch.Tensor) and np.array_equal(dev.cpu().numpy(), g[f"ci_{i}"])
        # column tiles smaller than the array (several uploads)
        assert np.array_equal(U.credible_interval_range(chain, max_bytes=8 * n * 40), g[f"ci_{i}"])
    maps = U.wavelet_credible_interval_range(make_chain(*CASES[0]), 10, 2, 2)
    assert [list(m.shape) for m in maps] == g["wav_shapes"].tolist()
    assert np.array_equal(np.concatenate([m.ravel() for m in maps]), g["wav_flat"])
    logpis = -np.abs(make_chain(1, 400, 14)[0])
    assert U.credible_region_threshold(logpis) == g["threshold"] and U.credible_region_threshold(logpis, alpha=0.2) == g["threshold20"]
    assert U.in_credible_region(g["threshold"] - 1.0, g["threshold"]) and not U.in_credible_region(g["threshold"] + 1.0, g["threshold"])
    with pytest.raises(TypeError):
        U.credible_interval_range(make_chain(8, 4, 1) + 1j)


def test_chain_to_pixels_is_the_batched_synthesis(px):
    """the plot scripts' per-sample transform.inverse loop (experiments/earthtopography/plot.py:103-109)
    as batched launches: real part of Psi(sample) against the oracle"""
    from oracle import pxmcmc_ref as R
    from pxmcmc_b200 import uncertainty as U

    L, B, J = 10, 2.0, 2
    t = px.transforms.SphericalWaveletTransform(L, B, J)
    ref = R.WaveletTransform(L, B, J)
    chain = np.random.default_rng(3).standard_normal((7, t.ncoefs))
    pix = U.chain_to_pixels(chain, t, batch=3)
    assert pix.shape == (7, L * (2 * L - 1)) and pix.dtype == np.float64
    for i in range(7):
        assert rel_l2(pix[i], ref.inverse(chain[i].astype(complex)).real) < TOL


def test_weaklensing_harmonic_fusion_equals_pixel_space_composition(px):
    """Phi(Psi X) and Psi^dagger(Phi^dagger r) through harmonic space against the literal composition through pixel
    space at L = 96 with a mask, batch of 3 chains; the harmonic ends of the synthesis pair are an adjoint pair"""
    import torch

    from pxmcmc_b200 import device as D

    L, B, J = 96, 2.0, 2
    rng = np.random.default_rng(23)
    mask = rng.random((L, 2 * L - 1)) > 0.3
    ngal = rng.uniform(10, 40, size=(L, 2 * L - 1))
    wl = px.measurements.WeakLensing(L, mask=mask, ngal=ngal)
    t = px.transforms.SphericalWaveletTransform(L, B, J, nchains=3)
    data = rng.standard_normal(wl.ndata) + 1j * rng.standard_normal(wl.ndata)
    fo = px.forward.ForwardOperator(data, 1 / wl.inv_cov, "synthesis", transform=t, measurement=wl, nparams=t.ncoefs)
    X = D.to_dev_c(rng.standard_normal((3, t.ncoefs)) + 1j * rng.standard_normal((3, t.ncoefs)))
    fused_p = fo.forward(X)
    fused_g = fo.calc_gradg(fused_p)
    fo.fuse_harmonic = False
    plain_p = fo.forward(X)
    plain_g = fo.calc_gradg(plain_p)
    assert rel_l2(D.to_host(fused_p), D.to_host(plain_p)) < 1e-12
    assert rel_l2(D.to_host(fused_g), D.to_host(plain_g)) < 1e-12
    x1 = rng.standard_normal(t.ncoefs) + 1j * rng.standard_normal(t.ncoefs)
    y1 = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    a = np.vdot(y1, t._inverse_harmonic(x1))
    b = np.vdot(t._inverse_adjoint_harmonic(y1), x1)
    assert abs(a - b) / abs(a) < TOL


@pytest.mark.parametrize("setting", ["analysis", "synthesis"])
def test_pxmala_device_resident_loop_equals_the_host_synchronised_loop(px, setting, monkeypatch):
    """PxMALA with the accept test, the step-size tuning and the state hand-over on the device (no host round trip per
    iteration) against the loop that decides on the host, fed the same Philox proposals and the same uniforms: identical
    acceptance trace, same step sizes, same tracked samples"""
    L, B, J = 16, 2.0, 2
    rng = np.random.default_rng(41)
    data = rng.standard_normal(L * (2 * L - 1)) + 0j
    runs = []
    for device_loop in (True, False):
        op = px.forward.SphericalWaveletTransformOperator(data, 0.05, setting, L, B, J)
        # a step of the order of the noise variance: both accepted and rejected proposals occur
        p = px.mcmc.PxMCMCParams(nsamples=5, nburn=4, ngap=2, delta=2e-3, lmda=1e-2, mu=2.0, verbosity=0,
                                 track=["logposterior", "L2", "prior", "chain", "predictions"])
        if setting == "analysis":
            reg = px.prior.L1("analysis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu)
        else:
            reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu, L=L, B=B, J_min=J)
        m = px.mcmc.PxMALA(op, reg, p, tune_delta=True, noise="device", seed=77, stream0=2)
        assert m._device_resident()
        start = np.random.default_rng(3).laplace(size=op.nparams) * 0.1
        if not device_loop:
            monkeypatch.setattr(m, "_device_resident", lambda: False)
            steps = iter(range(1, 10 ** 6))
            monkeypatch.setattr(np.random, "rand", lambda: _philox_uniform(77, 2, next(steps)))
        m.run(start)
        runs.append(m)
    a, b = runs
    assert 0 < sum(a.acceptance_trace) < len(a.acceptance_trace)  # both branches exercised
    assert a.acceptance_trace == b.acceptance_trace
    assert np.allclose(a.deltas_trace, b.deltas_trace, rtol=1e-12, atol=0)
    assert rel_l2(a.chain, b.chain) < TOL and rel_l2(a.preds, b.preds) < TOL
    assert rel_l2(a.logPi, b.logPi) < TOL and rel_l2(a.L2s, b.L2s) < TOL and rel_l2(a.priors, b.priors) < TOL


def test_skrock_device_noise_graph_replay_equals_eager_steps(px):
    """SKROCK with Philox normals: the step captured as one CUDA graph (device-side step counter) reproduces the
    eagerly launched step bit for bit, and the Philox normals are those of the update kernel's stream"""
    import torch

    from pxmcmc_b200 import device as D

    L, B, J, s_ = 12, 2.0, 2, 4
    rng = np.random.default_rng(8)
    npix = L * (2 * L - 1)
    A = sparse.random(40, npix, density=0.05, random_state=3, format="csr")
    y = rng.standard_normal(40)
    prm = px.mcmc.PxMCMCParams(delta=1e-7, lmda=5e-8, mu=1.0, s=s_, verbosity=0, nsamples=3, nburn=1, ngap=1,
                               track=["logposterior", "L2", "prior", "chain"])

    def make():
        op = px.forward.PathIntegralOperator(A, y, 0.1, "synthesis", L, B, J)
        reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-8, L=L, B=B, J_min=J)
        return px.mcmc.SKROCK(op, reg, prm, noise="device", seed=11, stream0=1), op

    m1, op = make()
    m2, _ = make()
    X0 = D.to_dev_c(rng.laplace(size=(1, op.nparams)) * 0.01)
    g = m2.capture(X0)
    xs = X0
    for _ in range(3):
        m1._step_counter = m2._step_counter
        xs = m1._chain_step_dev(xs)
        g.step()
        assert torch.equal(g.state()[0], xs)
        assert torch.equal(g.state()[1], D.to_dev_c(m1._forward_dev(xs)))
    # element e of the normal vector = normal (e & 1) of pair e >> 1 of the step's stream
    z = D.philox_normal_dev(2, 7, 11, step=5, stream0=1)
    z2 = D.philox_normal_dev(1, 7, 11, step=5, stream0=2)
    assert torch.equal(z[1], z2[0]) and not torch.equal(z[0], z[1])
    assert abs(float(D.philox_normal_dev(1, 200000, 3, step=1).mean())) < 0.01
    # run() with device noise uses the graph and fills the tracked arrays
    m3, _ = make()
    m3.run(D.to_host(X0[0]).real)
    assert np.isfinite(m3.logPi).all() and m3.chain.shape == (3, op.nparams)


def test_pxmala_batched_chains_equal_single_chain_samplers(px):
    """several PxMALA chains as one batch (per-chain step size, accept flag and uniform on the device): chain c is the
    chain a single-chain sampler with Philox stream stream0 + c produces"""
    L, B, J, nch = 16, 2.0, 2, 3
    rng = np.random.default_rng(43)
    data = rng.standard_normal(L * (2 * L - 1)) + 0j
    p = px.mcmc.PxMCMCParams(nsamples=4, nburn=3, ngap=2, delta=2e-3, lmda=1e-2, mu=2.0, verbosity=0,
                             track=["logposterior", "L2", "prior", "chain"])
    start = np.random.default_rng(3).laplace(size=L * (2 * L - 1)) * 0.1

    def sampler(nchains, stream0):
        op = px.forward.SphericalWaveletTransformOperator(data, 0.05, "analysis", L, B, J, nchains=nchains)
        reg = px.prior.L1("analysis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu)
        return px.mcmc.PxMALA(op, reg, p, tune_delta=True, noise="device", seed=5, stream0=stream0, nchains=nchains)

    batch = sampler(nch, 10)
    batch.run(start)
    assert batch.chain.shape == (nch, 4, start.size) and batch.acceptance_trace.shape[0] == nch
    traces = set()
    for c in range(nch):
        one = sampler(1, 10 + c)
        one.run(start)
        n = len(one.acceptance_trace)
        assert list(batch.acceptance_trace[c][:n]) == one.acceptance_trace
        assert np.allclose(batch.deltas_trace[c][: n + 1], one.deltas_trace, rtol=1e-13, atol=0)
        assert rel_l2(batch.chain[c], one.chain) < TOL and rel_l2(batch.logPi[c], one.logPi) < TOL
        traces.add(tuple(one.acceptance_trace[:6]))
    assert not np.allclose(batch.chain[0], batch.chain[1])
    with pytest.raises(NotImplementedError):
        px.mcmc.PxMALA(batch.forward, batch.prior, p, nchains=2)  # host-noise parity mode is single-chain


@pytest.mark.parametrize("noise", ["host", "device"])
def test_myula_checkpoint_resume_continues_the_same_chain(px, noise, tmp_path):
    """a run interrupted after a checkpoint and resumed by a NEW sampler object gives the chain of the uninterrupted
    run bit for bit: Philox steps (device noise, CUDA-graph replay) or numpy's global RNG stream (host noise)"""
    L, B, J = 12, 2.0, 2
    rng = np.random.default_rng(9)
    data = rng.standard_normal(L * (2 * L - 1)) + 0j
    track = ["logposterior", "L2", "prior", "chain", "predictions"]

    def sampler(nsamples):
        op = px.forward.SphericalWaveletTransformOperator(data, 0.2, "synthesis", L, B, J)
        p = px.mcmc.PxMCMCParams(nsamples=nsamples, nburn=2, ngap=3, delta=1e-5, lmda=2e-5, mu=1.0, verbosity=0, track=track)
        reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda, L=L, B=B, J_min=J)
        return px.mcmc.MYULA(op, reg, p, noise=noise, seed=21, stream0=4)

    start = np.random.default_rng(1).laplace(size=sampler(1).forward.nparams)
    np.random.seed(77)
    full = sampler(6)
    full.run(start)
    # the same run, stopped after 3 samples (checkpoint at the end of the shorter run) ...
    np.random.seed(77)
    first = sampler(6)
    first.nsamples = 3  # stop early; the tracked arrays keep their full length
    ck = str(tmp_path / "ck.npz")
    first.run(start, checkpoint=ck, checkpoint_every=4)
    # ... and continued by a new object from the file alone (the global RNG is clobbered in between)
    np.random.seed(12345)
    second = sampler(6)
    second.run(resume=ck)
    assert np.array_equal(second.chain, full.chain) and np.array_equal(second.logPi, full.logPi)
    assert np.array_equal(second.preds, full.preds) and np.array_equal(second.L2s, full.L2s)


def test_skrock_batched_chains_equal_single_chain_steps(px):
    """SKROCK steps of a batch of chains (Philox normals, stream stream0 + c per chain) = the single-chain steps"""
    import torch

    from pxmcmc_b200 import device as D

    L, B, J, s_, nch = 12, 2.0, 2, 3, 3
    rng = np.random.default_rng(18)
    npix = L * (2 * L - 1)
    A = sparse.random(30, npix, density=0.05, random_state=4, format="csr")
    y = rng.standard_normal(30)
    prm = px.mcmc.PxMCMCParams(delta=1e-7, lmda=5e-8, mu=1.0, s=s_, verbosity=0, nsamples=1)

    def make(nchains, stream0):
        op = px.forward.PathIntegralOperator(A, y, 0.1, "synthesis", L, B, J, nchains=nchains)
        reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-8, L=L, B=B, J_min=J)
        return px.mcmc.SKROCK(op, reg, prm, noise="device", seed=2, stream0=stream0, nchains=nchains), op

    mb, op = make(nch, 20)
    X0 = D.to_dev_c(rng.laplace(size=(nch, op.nparams)) * 0.01)
    mb._step_counter = 6
    Xb = mb._chain_step_dev(X0)
    for c in range(nch):
        m1, _ = make(1, 20 + c)
        m1._step_counter = 6
        assert torch.equal(m1._chain_step_dev(X0[c:c + 1])[0], Xb[c])
