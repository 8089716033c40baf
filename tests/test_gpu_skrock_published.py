"""GPU tests of SKROCK(scheme="published") and of the fused stage kernels both schemes run (`pxm_skrock_shift`,
`pxm_skrock_stage`): step parity with the oracle's published recursion (oracle/skrock_ref.py), the fused kernels
against the gradlogpi + lincomb composition they replace, device noise (graphs, batched chains), the stationary law on
a diagonal Gaussian target, a long run at the config-3 shape, and checkpoints."""
import numpy as np
import pytest
from scipy import sparse

from conftest import golden, rel_l2

pytestmark = pytest.mark.gpu

TOL = 1e-10


@pytest.fixture(scope="module")
def px():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pxmcmc_b200 import device, forward, mcmc, measurements, paths, prior, transforms

    class NS:
        pass

    ns = NS()
    ns.D, ns.forward, ns.mcmc, ns.measurements, ns.paths, ns.prior, ns.transforms = (
        device, forward, mcmc, measurements, paths, prior, transforms)
    return ns


def _oracle_path_case(A, data, sig, L, B, J, lmda):
    from oracle import pxmcmc_ref as R

    t = R.WaveletTransform(L, B, J)
    op = R.ForwardOperator(data, sig, "synthesis", t, R.PathIntegral(A), t.ncoefs)
    return op, R.S2WaveletsL1PowerWeights("synthesis", t.inverse, t.inverse_adjoint, lmda, L, B, J, eta=1)


def _step_with(px, m, X, Z):
    """one step of `m` from the host vector X with the injected real normals Z"""
    D = px.D
    return D.to_host(m._chain_step_dev(m._state(X), Z=D.to_dev_f(Z).reshape(1, -1))[0])


# ------------------------------------------------------------------ step parity against the oracle
@pytest.mark.parametrize("s", [1, 3, 5])
def test_published_step_golden_operator(px, s):
    from oracle import skrock_ref as S

    g = golden("ref_skrock_L10.npz")
    L, B, J = int(g["L"]), float(g["B"]), int(g["J_min"])
    A = sparse.csr_matrix((g["A_data"], g["A_indices"], g["A_indptr"]), shape=tuple(g["A_shape"]))
    delta, lmda, mu = float(g["delta"]), float(g["lmda"]), float(g["mu"])
    op = px.forward.PathIntegralOperator(A, g["data"], g["sig_d"], "synthesis", L, B, J)
    prm = px.mcmc.PxMCMCParams(delta=delta, lmda=lmda, mu=mu, s=s, verbosity=0, nsamples=1, track=[])
    reg = px.prior.S2_Wavelets_L1_Power_Weights("synthesis", op.transform.inverse, op.transform.inverse_adjoint,
                                               lmda * mu, L=L, B=B, J_min=J, eta=1)
    m = px.mcmc.SKROCK(op, reg, prm, scheme="published")
    Z = np.random.default_rng(s).standard_normal(op.nparams)
    Xn = _step_with(px, m, g["X"], Z)
    oop, opr = _oracle_path_case(A, g["data"], g["sig_d"], L, B, J, lmda * mu)
    Xo = S.skrock_step_published(oop, opr, delta, lmda, s, g["X"], Z)
    assert rel_l2(Xn, Xo) < TOL, f"s={s}: {rel_l2(Xn, Xo):.2e}"
    if s > 1:  # the schemes differ from stage 2 on
        assert rel_l2(_step_with(px, px.mcmc.SKROCK(op, reg, prm), g["X"], Z), Xo) > 1e-6


def test_published_step_complex(px):
    from oracle import pxmcmc_ref as R
    from oracle import skrock_ref as S

    L, B, J, s_ = 10, 2.0, 2, 3
    rng = np.random.default_rng(12)
    data = rng.standard_normal(L * (2 * L - 1)) + 1j * rng.standard_normal(L * (2 * L - 1))
    op = px.forward.SphericalWaveletTransformOperator(data, 0.2, "synthesis", L, B, J)
    prm = px.mcmc.PxMCMCParams(delta=1e-6, lmda=5e-7, mu=1.0, s=s_, complex=True, verbosity=0, nsamples=1, track=[])
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-7, L=L, B=B, J_min=J)
    m = px.mcmc.SKROCK(op, reg, prm, scheme="published")
    X = rng.laplace(size=op.nparams) + 1j * rng.laplace(size=op.nparams)
    np.random.seed(4)
    Z = np.random.randn(op.nparams) + 1j * np.random.randn(op.nparams)
    np.random.seed(4)
    Xn = m.chain_step(X)  # host noise: real part first, then imaginary
    t = R.WaveletTransform(L, B, J)
    oop = R.ForwardOperator(data, 0.2, "synthesis", t, R.IdentityMeasurement(data.size, data.size), t.ncoefs)
    oprior = R.S2WaveletsL1("synthesis", t.inverse, t.inverse_adjoint, 5e-7, L, B, J)
    assert rel_l2(Xn, S.skrock_step_published(oop, oprior, 1e-6, 5e-7, s_, X, Z)) < TOL


@pytest.fixture(scope="module")
def config3(px):
    """bench's config 3: 10^4 great circles between random end points (seed 7) rasterised on the device, L = 128"""
    L, B = 128, 2
    rng = np.random.default_rng(7)
    z = rng.uniform(-1, 1, size=(10000, 2))
    lon = rng.uniform(-180, 180, size=(10000, 2))
    lat = np.degrees(np.arcsin(z))
    A = px.paths.get_path_matrix(np.stack([lat[:, 0], lon[:, 0]], 1), np.stack([lat[:, 1], lon[:, 1]], 1), L)
    truth = np.random.default_rng(8).standard_normal(L * (2 * L - 1))
    y = A @ truth + 0.05 * rng.standard_normal(A.shape[0])
    return A, y, np.full(A.shape[0], 0.05), L, B, 2


def _config3_sampler(px, case, nchains=1, **kw):
    A, y, sig, L, B, J = case
    op = px.forward.PathIntegralOperator(A, y, sig, "synthesis", L, B, J, nchains=nchains)
    prm = px.mcmc.PxMCMCParams(delta=1e-6, lmda=5e-7, mu=1.0, s=10, verbosity=0, nsamples=1, track=[])
    reg = px.prior.S2_Wavelets_L1_Power_Weights("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-7,
                                               L=L, B=B, J_min=J, eta=1)
    return px.mcmc.SKROCK(op, reg, prm, scheme="published", nchains=nchains, **kw), op, reg


def test_published_step_config3(px, config3):
    from oracle import skrock_ref as S

    A, y, sig, L, B, J = config3
    m, op, reg = _config3_sampler(px, config3)
    assert op.nparams == 76068
    rng = np.random.default_rng(9)
    X = rng.laplace(size=op.nparams) * 1e-2
    Z = rng.standard_normal(op.nparams)
    Xn = _step_with(px, m, X, Z)
    oop, opr = _oracle_path_case(A, y, sig, L, B, J, 5e-7)
    assert rel_l2(reg.T, opr.T) < 1e-13
    Xo = S.skrock_step_published(oop, opr, 1e-6, 5e-7, 10, X, Z)
    assert np.isfinite(Xn).all() and rel_l2(Xn, Xo) < TOL, f"{rel_l2(Xn, Xo):.2e}"


# ------------------------------------------------------------------ fused kernels = the composition they replace
def _composed_shift(D, X, cs, zr, zi):
    import torch

    if zi is None:
        return D.lincomb_dev([(1.0, X)], z=zr, cz=cs)
    return D.lincomb_dev([(1.0, X), (cs, torch.complex(zr, zi))])


def _composed_stage1(D, X, gradg, prox, Tv, Ts, lmda, a, cs, e, zr, zi):
    import torch

    g = D.gradlogpi_dev(_composed_shift(D, X, cs, zr, zi), prox, Tv, Ts, gradg, lmda)
    if zi is None:
        return D.lincomb_dev([(1.0, X), (a, g)], z=zr, cz=e)
    return D.lincomb_dev([(1.0, X), (a, g), (e, torch.complex(zr, zi))])


@pytest.mark.parametrize("nch", [1, 3, 64, 65])
def test_fused_stages_equal_the_composed_kernels(px, nch):
    import torch

    D = px.D
    n, lmda, seed, step, stream0 = 1001, 0.7, 13, 5, 3
    gen = torch.Generator(device="cuda").manual_seed(nch)

    def cn(*shape):
        return torch.complex(torch.randn(*shape, dtype=torch.float64, device="cuda", generator=gen),
                             torch.randn(*shape, dtype=torch.float64, device="cuda", generator=gen))

    U, V, gradg, given = cn(nch, n), cn(nch, n), cn(nch, n) * 0.3, cn(nch, n)
    Tvec = torch.rand(n, dtype=torch.float64, device="cuda", generator=gen)
    zr_inj = torch.randn(nch, n, dtype=torch.float64, device="cuda", generator=gen)
    zi_inj = torch.randn(nch, n, dtype=torch.float64, device="cuda", generator=gen)
    z2 = D.philox_normal_dev(nch, 2 * n, seed, step, stream0)
    noises = {
        "injected real": (D.SkrockNoise(zr_inj), zr_inj, None),
        "injected complex": (D.SkrockNoise(zr_inj, zi_inj), zr_inj, zi_inj),
        "philox real": (D.SkrockNoise(seed=seed, step=step, stream0=stream0), D.philox_normal_dev(nch, n, seed, step,
                                                                                                  stream0), None),
        "philox complex": (D.SkrockNoise(complex=True, seed=seed, step=step, stream0=stream0),
                           z2[:, :n].contiguous(), z2[:, n:].contiguous()),
    }
    dstep = torch.full((1,), step, dtype=torch.int64, device="cuda")
    noises["philox complex, device step"] = (D.SkrockNoise(complex=True, seed=seed, step=999, stream0=stream0,
                                                           dstep=dstep), z2[:, :n].contiguous(), z2[:, n:].contiguous())
    a, b, cs, e = 0.31, 1.7, 0.45, 0.9
    for pname, (prox, Tv, Ts) in {"vector T": (None, Tvec, 0.0), "scalar T": (None, None, 0.6),
                                  "given prox": (given, None, 0.0)}.items():
        for zname, (Z, zr, zi) in noises.items():
            tag = f"{pname}, {zname}, {nch} chains"
            assert torch.equal(D.skrock_shift_dev(U, cs, Z), _composed_shift(D, U, cs, zr, zi)), tag
            got = D.skrock_stage_dev(U, None, gradg, prox, Tv, Ts, lmda, a, 1.0, 0.0, 0.0, Z=Z, c_shift=cs, e=e)
            assert torch.equal(got, _composed_stage1(D, U, gradg, prox, Tv, Ts, lmda, a, cs, e, zr, zi)), tag
        g = D.gradlogpi_dev(U, prox, Tv, Ts, gradg, lmda)
        for scheme, (c, c0) in {"reference": (-1.0, 1.0), "published": (-0.42, 0.0)}.items():
            want = D.lincomb_dev([(a, g), (b, U), (c, V)], c0=c0)
            got = D.skrock_stage_dev(U, V, gradg, prox, Tv, Ts, lmda, a, b, c, c0)
            assert torch.equal(got, want), f"{pname}, {scheme} stage j >= 2, {nch} chains"
            # in place, as the last stage of a captured step writes the state buffer (which may be V)
            Vc = V.clone()
            D.skrock_stage_dev(U, Vc, gradg, prox, Tv, Ts, lmda, a, b, c, c0, out=Vc)
            assert torch.equal(Vc, want)
    # the normals differ per chain (stream stream0 + chain) and the real and imaginary parts are different numbers
    Y = D.skrock_shift_dev(torch.zeros_like(U), 1.0, noises["philox complex"][0])
    assert torch.equal(Y.real, z2[:, :n]) and torch.equal(Y.imag, z2[:, n:])
    if nch > 1:
        assert not torch.equal(Y[0], Y[1])


# ------------------------------------------------------------------ device noise
def _small_path_case(px, nchains=1, complex=False, seed=11, stream0=1, s_=4, **kw):
    L, B, J = 12, 2.0, 2
    rng = np.random.default_rng(8)
    npix = L * (2 * L - 1)
    A = sparse.random(40, npix, density=0.05, random_state=3, format="csr")
    y = rng.standard_normal(40) + (1j * rng.standard_normal(40) if complex else 0)
    prm = px.mcmc.PxMCMCParams(delta=1e-7, lmda=5e-8, mu=1.0, s=s_, complex=complex, verbosity=0, **kw)
    op = px.forward.PathIntegralOperator(A, y, 0.1, "synthesis", L, B, J, nchains=nchains)
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-8, L=L, B=B, J_min=J)
    return px.mcmc.SKROCK(op, reg, prm, scheme="published", noise="device", seed=seed, stream0=stream0,
                          nchains=nchains), op


@pytest.mark.parametrize("complex_", [False, True])
def test_published_graph_replay_equals_eager_steps(px, complex_):
    import torch

    D = px.D
    m1, op = _small_path_case(px, complex=complex_, nsamples=3, nburn=1, ngap=1)
    m2, _ = _small_path_case(px, complex=complex_, nsamples=3, nburn=1, ngap=1)
    X0 = D.to_dev_c(np.random.default_rng(8).laplace(size=(1, op.nparams)) * 0.01)
    g = m2.capture(X0)
    xs = X0
    for _ in range(3):
        m1._step_counter = m2._step_counter
        xs = m1._chain_step_dev(xs)
        g.step()
        assert torch.equal(g.state()[0], xs)
        assert torch.equal(g.state()[1], D.to_dev_c(m1._forward_dev(xs)))
    if complex_:
        assert float(xs.imag.abs().max()) > 0


def test_published_batched_chains_equal_single_chain_steps(px):
    import torch

    D = px.D
    nch = 3
    mb, op = _small_path_case(px, nchains=nch, stream0=20, s_=3, nsamples=1)
    X0 = D.to_dev_c(np.random.default_rng(18).laplace(size=(nch, op.nparams)) * 0.01)
    mb._step_counter = 6
    Xb = mb._chain_step_dev(X0)
    for c in range(nch):
        m1, _ = _small_path_case(px, nchains=1, stream0=20 + c, s_=3, nsamples=1)
        m1._step_counter = 6
        assert torch.equal(m1._chain_step_dev(X0[c:c + 1])[0], Xb[c])


# ------------------------------------------------------------------ it samples
def test_published_scheme_samples_a_stiff_diagonal_gaussian(px):
    """grad log pi(x) = -a (x - d) per coordinate, a log-spaced over [1, 1000], s = 10, delta = 0.15 (a_max delta = 150,
    the limit is 193.6): the pooled mean is d and the pooled variance is the scheme's exact stationary variance
    S^2 / (1 - R^2), which differs from 1/a at the stiff end"""
    from oracle import skrock_ref as S

    n, nch, s, delta = 1024, 4096, 10, 0.15
    a = np.logspace(0, 3, n)
    d = np.random.default_rng(5).standard_normal(n)
    t = px.transforms.IdentityTransform()
    op = px.forward.ForwardOperator(d, 1 / np.sqrt(a), "synthesis", t, px.measurements.Identity(n, n), nparams=n)
    reg = px.prior.L1("synthesis", t.inverse, t.inverse_adjoint, 0.0)
    prm = px.mcmc.PxMCMCParams(delta=delta, lmda=1.0, mu=1.0, s=s, nsamples=64, nburn=200, ngap=20, verbosity=0,
                               track=[])
    m = px.mcmc.SKROCK(op, reg, prm, scheme="published", noise="device", seed=3, nchains=nch, summarise=("chain",))
    assert a.max() * delta < m.stability_limit
    m.run(np.zeros(n))
    sm = m.summary["chain"]
    R, Sx = S.scalar_step(a, d, delta, s)
    var_exact = Sx ** 2 / (1 - R ** 2)
    assert np.abs(var_exact * a - 1).max() > 0.05  # the stiff coordinates are visibly not at 1/a
    assert np.all(np.abs(sm.mean - d) < 6 * sm.mcse), np.abs((sm.mean - d) / sm.mcse).max()
    assert np.all(np.abs(sm.var / var_exact - 1) < 0.02), np.abs(sm.var / var_exact - 1).max()


def test_published_long_run_config3_stays_bounded(px, config3):
    """1000 graphed steps of 8 chains at bench's config 3 (delta = 1e-6, lmda = 5e-7) from zero: log pi finite and
    max |X| < 10 throughout (the reference scheme passes 1e70 within a few steps)"""
    import torch

    D = px.D
    m, op, _ = _config3_sampler(px, config3, nchains=8, noise="device", seed=5)
    g = m.capture(D.to_dev_c(np.zeros((8, op.nparams))))
    worst = torch.zeros((), dtype=torch.float64, device="cuda")
    lps = []
    for i in range(1000):
        g.step()
        X, P = g.state()
        worst = torch.maximum(worst, X.abs().max())
        if i % 10 == 9:
            lps.append(m._logpi_dev(X, P)[0])
    assert float(worst) < 10
    assert np.isfinite(np.concatenate(lps)).all()


# ------------------------------------------------------------------ checkpoints
@pytest.mark.parametrize("noise", ["device", "host"])
def test_published_checkpoint_resume_and_scheme_mismatch(px, noise, tmp_path):
    L, B, J, s_ = 12, 2.0, 2, 3
    rng = np.random.default_rng(8)
    A = sparse.random(40, L * (2 * L - 1), density=0.05, random_state=3, format="csr")
    y = rng.standard_normal(40)

    def make(nsamples, scheme="published"):
        prm = px.mcmc.PxMCMCParams(delta=1e-7, lmda=5e-8, mu=1.0, s=s_, verbosity=0, nsamples=nsamples, nburn=1, ngap=2,
                                   track=["logposterior", "L2", "prior", "chain", "predictions"])
        op = px.forward.PathIntegralOperator(A, y, 0.1, "synthesis", L, B, J)
        reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-8, L=L, B=B, J_min=J)
        return px.mcmc.SKROCK(op, reg, prm, scheme=scheme, noise=noise, seed=11, stream0=1)

    start = rng.laplace(size=make(1).forward.nparams) * 0.01
    np.random.seed(3)
    full = make(5)
    full.run(start)
    np.random.seed(3)
    first = make(5)
    first.nsamples = 2
    ck = str(tmp_path / "skrock.npz")
    first.run(start, checkpoint=ck, checkpoint_every=2)
    with np.load(ck) as f:
        assert str(f["scheme"]) == "published"
    np.random.seed(4242)
    second = make(5)
    second.run(resume=ck)
    assert np.array_equal(second.chain, full.chain) and np.array_equal(second.logPi, full.logPi)
    assert np.array_equal(second.preds, full.preds)
    with pytest.raises(ValueError, match="scheme"):
        make(5, "reference").run(resume=ck)
    # a checkpoint without the field was written by the reference scheme
    with np.load(ck) as f:
        old = {k: f[k] for k in f.files if k != "scheme"}
    legacy = str(tmp_path / "legacy.npz")
    np.savez(legacy, **old)
    with pytest.raises(ValueError, match="scheme"):
        make(5).run(resume=legacy)
    make(5, "reference").run(resume=legacy)
