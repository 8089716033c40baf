"""GPU tests of the MAP estimate and the step-size bound: `ForwardOperator.lipschitz()` against the eigenvalues of the
dense oracle matrix (oracle/map_ref.py) for every carried form of gradg, `pxm_fista_update` iterates against the numpy
FISTA, graph replay against the eager loop, the minimiser's optimality conditions, SKROCK(published) started at the
MAP at 0.9 max_stable_delta(), and the documented refusals."""
import numpy as np
import pytest
from scipy import sparse

from conftest import golden, rel_l2

pytestmark = pytest.mark.gpu

L, B, J = 10, 2.0, 2
NPIX = L * (2 * L - 1)
LIP_TOL = 1e-8


@pytest.fixture(scope="module")
def px():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pxmcmc_b200 import device, forward, mcmc, measurements, prior, transforms

    class NS:
        pass

    ns = NS()
    ns.D, ns.forward, ns.mcmc, ns.measurements, ns.prior, ns.transforms = (
        device, forward, mcmc, measurements, prior, transforms)
    return ns


def _data():
    return np.random.default_rng(0).standard_normal(NPIX)


def _sigma(case):
    rng = np.random.default_rng(5)
    return {"scalar": 0.3, "ring": np.repeat(rng.uniform(0.2, 0.5, L), 2 * L - 1),
            "pixel": rng.uniform(0.2, 0.5, NPIX)}[case]


def _oracle_wavelet(sig):
    from oracle import pxmcmc_ref as R

    t = R.WaveletTransform(L, B, J)
    return R.ForwardOperator(_data(), sig, "synthesis", t, R.IdentityMeasurement(NPIX, NPIX), t.ncoefs), t


_DENSE = {}


def _dense(key, make):
    from oracle import map_ref as M

    if key not in _DENSE:
        _DENSE[key] = M.dense_operator(make())
    return _DENSE[key]


def _lam(Mx):
    return np.linalg.eigvalsh(Mx)[-1]


# ------------------------------------------------------------------ 1. lipschitz() against the dense oracle
@pytest.mark.parametrize("case,gram,kind", [("scalar", True, "harm"), ("ring", True, "harm"), ("ring", False, "ring"),
                                            ("pixel", True, None)])
def test_lipschitz_wavelet_operator(px, case, gram, kind):
    """scalar sigma: Gram form; per-ring sigma: weighted Gram form, or ring form without it; pixel-varying sigma:
    forward + calc_gradg; then the literal composition, and the real-pairs operator"""
    sig = _sigma(case)

    def make():
        op = px.forward.SphericalWaveletTransformOperator(_data(), sig, "synthesis", L, B, J)
        op.fuse_gram = gram
        return op

    op = make()
    assert op._ring_kind() == kind
    want = _lam(_dense(case, lambda: _oracle_wavelet(sig)[0]))
    lam = op.lipschitz()
    assert abs(lam - want) <= LIP_TOL * want, (lam, want)
    assert op._lipschitz_cache[3] < 200  # ARPACK's matrix-vector products
    literal = make()
    literal.fuse_ring = literal.fuse_gram = False
    assert literal._ring_kind() is None
    assert abs(literal.lipschitz() - want) <= LIP_TOL * want
    paired = make().paired()  # (a fresh operator: nothing cached)
    assert abs(paired.lipschitz() - want) <= LIP_TOL * want


def test_lipschitz_path_integral_golden(px):
    from oracle import pxmcmc_ref as R

    g = golden("ref_skrock_L10.npz")
    Lg, Bg, Jg = int(g["L"]), float(g["B"]), int(g["J_min"])
    A = sparse.csr_matrix((g["A_data"], g["A_indices"], g["A_indptr"]), shape=tuple(g["A_shape"]))
    op = px.forward.PathIntegralOperator(A, g["data"], g["sig_d"], "synthesis", Lg, Bg, Jg)
    t = R.WaveletTransform(Lg, Bg, Jg)
    want = _lam(_dense("path", lambda: R.ForwardOperator(g["data"], g["sig_d"], "synthesis", t, R.PathIntegral(A),
                                                          t.ncoefs)))
    assert abs(op.lipschitz() - want) <= LIP_TOL * want


def _weaklensing(px, sig_complex=True):
    from oracle import pxmcmc_ref as R

    g = golden("ref_weaklensing_L12.npz")
    Lw = int(g["L"])
    wl = px.measurements.WeakLensing(Lw, mask=g["mask"], ngal=g["ngal"])
    sig = 1 / wl.inv_cov
    if sig_complex:
        sig = sig.astype(complex)
    t = px.transforms.SphericalWaveletTransform(Lw, 2, 2)
    op = px.forward.ForwardOperator(g["gdata"], sig, "synthesis", transform=t, measurement=wl, nparams=t.ncoefs)
    ot = R.WaveletTransform(Lw, 2, 2)
    oop = lambda: R.ForwardOperator(g["gdata"], sig, "synthesis", ot, R.WeakLensing(Lw, mask=g["mask"], ngal=g["ngal"]),  # noqa: E731
                                    ot.ncoefs)
    return op, oop, Lw


def test_lipschitz_weak_lensing_golden_complex_sigma(px):
    op, oop, _ = _weaklensing(px)
    assert np.iscomplexobj(op.data) and op._fused()
    want = _lam(_dense("wl", oop))
    assert abs(op.lipschitz() - want) <= LIP_TOL * want


def test_lipschitz_config1_device_matrix(px):
    """config 1 (L = 32, B = 1.5): eigvalsh of the matrix assembled from the device operator's own columns"""
    import torch

    D = px.D
    L1_, B1 = 32, 1.5
    data = np.random.default_rng(3).standard_normal(L1_ * (2 * L1_ - 1))
    op = px.forward.SphericalWaveletTransformOperator(data, 1.0, "synthesis", L1_, B1, 2)
    z = op._zero_data()
    n, nb = op.nparams, 64
    Mx = np.empty((n, n), dtype=complex)
    for c0 in range(0, n, nb):
        k = min(nb, n - c0)
        E = torch.zeros((k, n), dtype=D.CDT, device="cuda")
        E[torch.arange(k), torch.arange(c0, c0 + k)] = 1.0
        Mx[:, c0:c0 + k] = D.to_host(z._normal_apply(E)).T
    assert np.abs(Mx - Mx.conj().T).max() <= 1e-12 * np.abs(Mx).max()
    want = np.linalg.eigvalsh((Mx + Mx.conj().T) / 2)[-1]
    assert abs(op.lipschitz() - want) <= LIP_TOL * want


def _eigsh_other(op, ncv, seed):
    from scipy.sparse.linalg import LinearOperator, eigsh

    from pxmcmc_b200 import device as D

    z, n = op._zero_data(), op.nparams
    mv = lambda v: D.to_host(z._normal_apply(D.to_dev_c(np.ravel(v)).reshape(1, n))[0])  # noqa: E731
    rng = np.random.default_rng(seed)
    v0 = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    A = LinearOperator((n, n), matvec=mv, dtype=np.complex128)
    return float(eigsh(A, k=1, which="LA", tol=1e-12, ncv=ncv, v0=v0, return_eigenvectors=False)[0])


def test_lipschitz_config3_config4_against_eigsh(px):
    from pxmcmc_b200 import paths

    Lc, Bc = 128, 2
    rng = np.random.default_rng(7)
    z = rng.uniform(-1, 1, size=(10000, 2))
    lon = rng.uniform(-180, 180, size=(10000, 2))
    lat = np.degrees(np.arcsin(z))
    A = paths.get_path_matrix(np.stack([lat[:, 0], lon[:, 0]], 1), np.stack([lat[:, 1], lon[:, 1]], 1), Lc)
    y = A @ np.random.default_rng(8).standard_normal(A.shape[1]) + 0.05 * rng.standard_normal(A.shape[0])
    op3 = px.forward.PathIntegralOperator(A, y, np.full(A.shape[0], 0.05), "synthesis", Lc, Bc, 2)
    lam = op3.lipschitz()
    want = _eigsh_other(op3, 40, 1)
    assert abs(lam - want) <= LIP_TOL * want, (lam, want)
    op4 = _config4_operator(px)
    lam = op4.lipschitz()
    want = _eigsh_other(op4, 40, 2)
    assert abs(lam - want) <= LIP_TOL * want, (lam, want)


def _config4_operator(px):
    """config 4 on one GPU: weak lensing behind a wavelet synthesis at L = 512, masked, ngal = 30, sigma complex"""
    from test_gpu_configs import wl_mask

    L4 = 512
    wl = px.measurements.WeakLensing(L4, mask=wl_mask(L4), ngal=np.full((L4, 2 * L4 - 1), 30.0))
    tr = px.transforms.SphericalWaveletTransform(L4, 2.0, 2)
    rng = np.random.default_rng(11)
    data = rng.standard_normal(wl.ndata) + 1j * rng.standard_normal(wl.ndata)
    return px.forward.ForwardOperator(data, (1.0 / wl.inv_cov).astype(complex), "synthesis", transform=tr,
                                      measurement=wl, nparams=tr.ncoefs)


# ------------------------------------------------------------------ 2. FISTA iterates against the oracle
def _sampler(px, op, T, nchains=1, lmda=1e-4, mu=100.0, cls=None, **kw):
    prm = px.mcmc.PxMCMCParams(lmda=lmda, mu=mu, delta=1e-6, s=10, verbosity=0, nsamples=1, track=[])
    if T == "vector":
        reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, lmda * mu, L=L,
                                      B=B, J_min=J)
    else:
        reg = px.prior.L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, lmda * mu)
    return (cls or px.mcmc.MYULA)(op, reg, prm, nchains=nchains, **kw)


def _oracle_prior(T, lmda=1e-4, mu=100.0):
    from oracle import pxmcmc_ref as R

    t = R.WaveletTransform(L, B, J)
    if T == "vector":
        return R.S2WaveletsL1("synthesis", t.inverse, t.inverse_adjoint, lmda * mu, L, B, J)
    return R.L1("synthesis", t.inverse, t.inverse_adjoint, lmda * mu)


class _Dense:
    def __init__(self, op, Mx):
        from oracle import map_ref as M

        self.Mx, self.b = Mx, -M.gradg(op, np.zeros(op.nparams))

    def forward(self, x):
        return x

    def calc_gradg(self, x):
        return self.Mx @ x - self.b


def _device_iterates(px, m, X0, t, niter):
    """the iterates of pxm_fista_update driven by the sampler's own gradg, eagerly"""
    import torch

    D = px.D
    X = D.to_dev_c(X0).clone()
    Y = X.clone()
    state = torch.tensor([0.0, 1.0], dtype=D.FDT, device="cuda")
    hist = torch.zeros((7, X.shape[0], 2), dtype=D.FDT, device="cuda")
    Tv, Ts = m._fused_prox()
    out = []
    for k in range(niter):
        D.fista_update_dev(Y, m._gradg_at(Y), X, Tv, Ts, t / m.lmda, t, state, hist, out=(X, Y))
        out.append(D.to_host(X))
        dx2, x2 = D.to_host(hist[k % 7]).T
        assert np.allclose(x2, np.sum(np.abs(out[-1]) ** 2, axis=1), rtol=1e-12)
        prev = out[-2] if k else np.asarray(X0)
        assert np.allclose(dx2, np.sum(np.abs(out[-1] - prev) ** 2, axis=1), rtol=1e-9, atol=1e-300)
    assert D.to_host(state)[0] == niter
    return out


@pytest.mark.parametrize("T", ["vector", "scalar"])
@pytest.mark.parametrize("nch", [1, 3, 65])
def test_fista_iterates_match_the_oracle(px, T, nch):
    from oracle import map_ref as M

    op = px.forward.SphericalWaveletTransformOperator(_data(), 0.3, "synthesis", L, B, J, nchains=nch)
    m = _sampler(px, op, T, nchains=nch)
    t = 1.0 / op.lipschitz()
    X0 = np.random.default_rng(nch).laplace(size=(nch, op.nparams)) * 0.1
    got = _device_iterates(px, m, X0, t, 50)
    oop, _ = _oracle_wavelet(0.3)
    oprior = _oracle_prior(T)
    for c in range(nch):
        fwd = oop if c == 0 else _Dense(oop, _dense("scalar", lambda: oop))
        want = M.fista(fwd, oprior, m.lmda, t, X0[c], 50)
        err = max(rel_l2(g[c], w) for g, w in zip(got, want))
        assert err <= 1e-10, f"chain {c}: {err:.2e}"


def test_graph_replay_equals_eager_loop(px):
    import torch

    op = px.forward.SphericalWaveletTransformOperator(_data(), 0.3, "synthesis", L, B, J, nchains=3)
    X0 = np.random.default_rng(4).laplace(size=(3, op.nparams)) * 0.1
    graphed = _sampler(px, op, "vector", nchains=3)
    assert graphed._native()
    xg, ig = graphed.map_estimate(X0, tol=0.0, maxiter=120)  # two graph replays of 50, then 20 eager iterations
    eager = _sampler(px, op, "vector", nchains=3)
    eager._FISTA_BLOCK = 1000  # maxiter below the block: no graph
    xe, ie = eager.map_estimate(X0, tol=0.0, maxiter=120)
    assert ig["iterations"] == ie["iterations"] == 120 and not ig["converged"]
    assert np.array_equal(xg, xe)
    assert np.array_equal(ig["F"], ie["F"])
    ref = _device_iterates(px, graphed, X0, ig["step"], 120)[-1]
    assert torch.equal(torch.from_numpy(xg), torch.from_numpy(ref))


# ------------------------------------------------------------------ 3. optimality
def test_map_estimate_optimality(px):
    import torch

    D = px.D
    tol = 1e-8
    op = px.forward.SphericalWaveletTransformOperator(_data(), 0.3, "synthesis", L, B, J, nchains=3)
    m = _sampler(px, op, "vector", nchains=3)
    X0 = np.random.default_rng(6).laplace(size=(3, op.nparams)) * np.array([[0.01], [1.0], [10.0]])
    x, info = m.map_estimate(X0, tol=tol)
    assert info["converged"] and x.shape == (3, op.nparams)
    assert info["relative_change"].shape == (info["iterations"] // 50 + (info["iterations"] % 50 > 0), 3)
    t = info["step"]
    Tv, Ts = m._fused_prox()
    Xd = D.to_dev_c(x)

    def prox_grad(Z):
        return D.soft_dev(Z - t * m._gradg_at(Z), Tv * (t / m.lmda), 0.0)

    res = torch.linalg.vector_norm(Xd - prox_grad(Xd), dim=1) / torch.linalg.vector_norm(Xd, dim=1)
    assert float(res.max()) <= 10 * tol, D.to_host(res)
    # F at the estimate is no larger than after 10^4 proximal-gradient (ISTA) steps from the same starts
    Z = D.to_dev_c(X0)
    for _ in range(10_000):
        Z = prox_grad(Z)
    F_ista = D.to_host(m._map_objective(Z))
    F = np.asarray(info["F"])
    assert np.all(F <= F_ista * (1 + 1e-12)), (F, F_ista)
    assert np.allclose(F, D.to_host(m._map_objective(Xd)), rtol=0, atol=0)
    # three starts, one minimum
    assert (F.max() - F.min()) <= 1e-8 * F.min(), F
    # a 1-D start of a one-chain sampler gives a 1-D estimate, a valid start point of run()
    op1 = px.forward.SphericalWaveletTransformOperator(_data(), 0.3, "synthesis", L, B, J)
    m1 = _sampler(px, op1, "vector")
    x1, i1 = m1.map_estimate(X0[1], tol=tol)
    assert x1.shape == (op1.nparams,) and abs(i1["F"] - F[1]) <= 1e-8 * F[1]


# ------------------------------------------------------------------ 4. use: SKROCK(published) started at the MAP
def test_skrock_published_from_the_map_at_the_stability_bound(px):
    import torch

    from pxmcmc_b200 import paths

    D = px.D
    Lc, Bc = 128, 2
    rng = np.random.default_rng(7)
    z = rng.uniform(-1, 1, size=(10000, 2))
    lon = rng.uniform(-180, 180, size=(10000, 2))
    lat = np.degrees(np.arcsin(z))
    A = paths.get_path_matrix(np.stack([lat[:, 0], lon[:, 0]], 1), np.stack([lat[:, 1], lon[:, 1]], 1), Lc)
    y = A @ np.random.default_rng(8).standard_normal(A.shape[1]) + 0.05 * rng.standard_normal(A.shape[0])

    def make(nch, scheme="published", **kw):
        op = px.forward.PathIntegralOperator(A, y, np.full(A.shape[0], 0.05), "synthesis", Lc, Bc, 2, nchains=nch)
        prm = px.mcmc.PxMCMCParams(delta=1e-6, lmda=5e-7, mu=1.0, s=10, verbosity=0, nsamples=1, track=[])
        reg = px.prior.S2_Wavelets_L1_Power_Weights("synthesis", op.transform.inverse, op.transform.inverse_adjoint,
                                                   5e-7, L=Lc, B=Bc, J_min=2, eta=1)
        return px.mcmc.SKROCK(op, reg, prm, scheme=scheme, nchains=nch, **kw)

    one = make(1)
    x_map, info = one.map_estimate(np.zeros(one.forward.nparams), maxiter=2000)
    assert np.isfinite(x_map).all() and info["F_history"][-1, 0] <= info["F_history"][0, 0]
    m = make(8, noise="device", seed=5)
    m.delta = 0.9 * m.max_stable_delta()
    assert np.isfinite(m.delta) and m.delta > 0
    g = m.capture(D.to_dev_c(np.tile(x_map, (8, 1))))
    lps = []
    for i in range(1000):
        g.step()
        if i % 10 == 9:
            X, P = g.state()
            lps.append(m._logpi_dev(X, P)[0])
    assert np.isfinite(np.concatenate(lps)).all()
    assert bool(torch.isfinite(g.state()[0]).all())
    assert np.isnan(make(1, scheme="reference").max_stable_delta())


# ------------------------------------------------------------------ 5. refusals
def test_refusals(px):
    op = px.forward.SphericalWaveletTransformOperator(_data(), 0.3, "analysis", L, B, J)
    reg = px.prior.L1("analysis", op.transform.forward, op.transform.inverse, 1e-2)
    prm = px.mcmc.PxMCMCParams(lmda=1e-4, mu=100.0, verbosity=0, nsamples=1, track=[])
    m = px.mcmc.MYULA(op, reg, prm)
    for call in (m.map_estimate, m.max_stable_delta):
        with pytest.raises(NotImplementedError, match="analysis"):
            call()

    op = px.forward.SphericalWaveletTransformOperator(_data(), 0.3, "synthesis", L, B, J)

    class MyL1(px.prior.L1):
        def proxf(self, X):
            return super().proxf(X)

    m = px.mcmc.MYULA(op, MyL1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 1e-2), prm)
    for call in (m.map_estimate, m.max_stable_delta):
        with pytest.raises(NotImplementedError, match="prox"):
            call()

    opf = px.forward.SphericalWaveletTransformOperator(_data(), 0.3, "synthesis", L, B, J)
    # the state a 2-D sigma leaves: a general sparse inverse covariance and no diagonal
    opf.invcov, opf._diag = sparse.random(NPIX, NPIX, density=0.01, random_state=1, format="csr"), None
    m = _sampler(px, opf, "vector")
    for call in (m.map_estimate, m.max_stable_delta, opf.lipschitz):
        with pytest.raises(NotImplementedError, match="full covariance"):
            call()

    opc, _, Lw = _weaklensing(px, sig_complex=False)
    assert np.any(np.asarray(opc._diag).imag != 0)  # the reference's rule gave IC the phase -pi/4
    prm = px.mcmc.PxMCMCParams(lmda=1e-4, mu=1.0, verbosity=0, nsamples=1, track=[])
    reg = px.prior.S2_Wavelets_L1("synthesis", opc.transform.inverse, opc.transform.inverse_adjoint, 1e-4, L=Lw, B=2,
                                  J_min=2)
    for cls in (px.mcmc.MYULA, px.mcmc.SKROCK):
        kw = {"scheme": "published"} if cls is px.mcmc.SKROCK else {}
        m = cls(opc, reg, prm, **kw)
        for call in (m.map_estimate, m.max_stable_delta, opc.lipschitz):
            with pytest.raises(ValueError, match="complex array"):
                call()
