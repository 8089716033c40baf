"""GPU tests of the rank-normalised diagnostics (pxm_rank_diagnostics, diagnostics.rank_diagnostics) against the numpy
oracle (oracle/rank_diagnostics_ref.py): shapes from one chain of 4 samples up to the 16 384-sample limit, data with
long autocorrelation, heavy tails, unequal spread, an offset chain and heavy ties; NaN handling; bit-for-bit
invariances; an end-to-end MYULA run; refusals.

Bars: R-hat 1e-12 absolute, ESS 1e-10 relative (the device uses direct lag sums and normcdfinv, the oracle an FFT and
scipy's ndtri)."""
import numpy as np
import pytest

from oracle import rank_diagnostics_ref as K

pytestmark = pytest.mark.gpu

SENTINEL = -7.0


@pytest.fixture(scope="module")
def px():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pxmcmc_b200 import device, diagnostics

    class NS:
        pass

    ns = NS()
    ns.torch, ns.D, ns.diag = torch, device, diagnostics
    return ns


KINDS = ("iid", "ar09", "ar099", "cauchy", "unequal", "offset", "ties")


def make(kind, m, n, k, seed):
    rng = np.random.default_rng(seed)
    if kind in ("ar09", "ar099"):
        phi = 0.9 if kind == "ar09" else 0.99
        e = rng.standard_normal((m, n, k))
        x = np.empty_like(e)
        x[:, 0] = e[:, 0] / np.sqrt(1 - phi ** 2)
        for t in range(1, n):
            x[:, t] = phi * x[:, t - 1] + e[:, t]
        return x
    if kind == "cauchy":
        return rng.standard_cauchy((m, n, k))
    x = rng.standard_normal((m, n, k))
    if kind == "unequal":
        x[1::2] *= 2.0
    elif kind == "offset":
        x[m // 2] += 3.0
    elif kind == "ties":
        x = np.floor(x * 1.5)  # about 8 distinct values
    return x


def mixed(m, n, ncols, seed):
    """ncols columns cycling through KINDS"""
    x = np.empty((m, n, ncols))
    for i, kind in enumerate(KINDS):
        cols = np.arange(i, ncols, len(KINDS))
        if cols.size:
            x[:, :, cols] = make(kind, m, n, cols.size, seed + i)
    return x


def check(got, ref, what):
    for name, g, r in zip(("rhat", "ess_bulk", "ess_tail"), got, ref):
        g, r = np.asarray(g), np.asarray(r)
        assert not np.any(g == SENTINEL), f"{what} {name}: a column was never written"
        assert np.array_equal(np.isnan(g), np.isnan(r)), f"{what} {name}: NaN pattern"
        ok = ~np.isnan(r)
        if name == "rhat":
            fin = ok & np.isfinite(r)
            assert np.array_equal(g[ok & ~fin], r[ok & ~fin]), f"{what} {name}: inf"
            d = np.abs(g[fin] - r[fin])
            assert np.all(d <= 1e-12), f"{what} {name}: worst {d.max()}"
        else:
            d = np.abs(g[ok] - r[ok]) / np.abs(r[ok])
            assert np.all(d <= 1e-10), f"{what} {name}: worst {d.max()} at {np.argmax(d)}"


def abi(px, x):
    """pxm_rank_diagnostics on a host array [m, n, ncols], outputs pre-filled with a sentinel"""
    from pxmcmc_b200._lib import check as ok, lib, ptr, stream_ptr

    torch = px.torch
    m, n, ncols = x.shape
    xd = torch.from_numpy(np.ascontiguousarray(x.reshape(m * n, ncols))).to(px.D.dev())
    scratch = torch.full((lib.pxm_rank_diagnostics_scratch_doubles(m, n, ncols),), np.nan, dtype=torch.float64,
                         device=xd.device)
    out = torch.full((3, ncols), SENTINEL, dtype=torch.float64, device=xd.device)
    ok(lib.pxm_rank_diagnostics(ptr(xd), m, n, ncols, ncols, ptr(scratch), ptr(out[0]), ptr(out[1]), ptr(out[2]),
                                stream_ptr()))
    return out.cpu().numpy()


SHAPES = [((1, 4), 1000), ((1, 5), 33), ((2, 7), 31), ((3, 17), 1000), ((4, 100), 33), ((4, 101), 1000),
          ((64, 256), 31), ((8, 2048), 33)]


@pytest.mark.parametrize("mn,ncols", SHAPES, ids=[f"{a}x{b}-{c}" for (a, b), c in SHAPES])
def test_against_oracle(px, mn, ncols):
    m, n = mn
    x = mixed(m, n, ncols, seed=m * 1000 + n)
    check(abi(px, x), K.rank_diagnostics(x), f"{m}x{n}")


@pytest.mark.parametrize("mn", [(1, 4), (4, 101), (64, 256), (8, 2048)])
def test_one_column_and_every_kind_at_the_limit(px, mn):
    m, n = mn
    for i, kind in enumerate(KINDS):
        x = make(kind, m, n, 1, seed=7 + i)
        check(abi(px, x), K.rank_diagnostics(x), f"{kind} {m}x{n}")


def test_constant_and_non_finite_columns(px):
    rng = np.random.default_rng(11)
    for m, n in ((3, 9), (4, 100), (8, 2048)):
        x = rng.standard_normal((m, n, 8))
        x[:, :, 0] = 1.25
        x[1, n // 2, 2] = np.nan
        x[0, 0, 4] = np.inf
        x[m - 1, n - 1, 5] = -np.inf
        got = abi(px, x)
        h = n // 2
        assert np.isnan(got[0, 0]) and got[1, 0] == 2 * m * h and got[2, 0] == 2 * m * h
        assert np.all(np.isnan(got[:, [2, 4, 5]]))
        assert np.all(np.isfinite(got[:, [1, 3, 6, 7]]))
        check(got, K.rank_diagnostics(x), f"special {m}x{n}")
    # n < 4: every column NaN
    assert np.all(np.isnan(abi(px, rng.standard_normal((40, 3, 5)))))


def test_invariances_bit_for_bit(px):
    rd = px.diag.rank_diagnostics
    x = mixed(8, 300, 64, seed=21)
    base = rd(x)
    for a, b in zip(rd(x * 2.0 ** 20), base):
        assert np.array_equal(a, b, equal_nan=True)
    y = np.random.default_rng(22).standard_normal((8, 300, 64))
    assert np.array_equal(rd(np.exp(y)).ess_bulk, rd(y).ess_bulk)
    for a, b in zip(rd(x, max_bytes=1), base):  # 32 columns per block
        assert np.array_equal(a, b, equal_nan=True)


def test_numpy_tensor_memmap_agree(px, tmp_path):
    torch = px.torch
    rd = px.diag.rank_diagnostics
    x = mixed(6, 50, 40, seed=31)
    base = rd(x)
    mm = np.lib.format.open_memmap(tmp_path / "chain.npy", mode="w+", dtype=np.float64, shape=x.shape)
    mm[:] = x
    mm.flush()
    ro = np.load(tmp_path / "chain.npy", mmap_mode="r")
    t = rd(torch.from_numpy(x).to(px.D.dev()))
    assert all(isinstance(v, torch.Tensor) and v.is_cuda for v in t)
    for got in (rd(ro), tuple(v.cpu().numpy() for v in t)):
        for a, b in zip(got, base):
            assert np.array_equal(a, b, equal_nan=True)
    # one chain as [nsamples, nparams]
    for a, b in zip(rd(x[2]), K.rank_diagnostics(x[2:3])):
        assert np.allclose(a, b, rtol=1e-10, atol=1e-12, equal_nan=True)
    check(base, K.rank_diagnostics(x), "api")


def test_myula_tracked_chain_end_to_end(px):
    from pxmcmc_b200 import forward, mcmc, prior, sht

    L, B, J, nch = 16, 1.5, 2, 8
    rng = np.random.default_rng(12)
    flm = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    data = sht.inverse(flm, L).ravel()
    op = forward.SphericalWaveletTransformOperator(data, 0.3, "synthesis", L, B, J, nchains=nch)
    p = mcmc.PxMCMCParams(nsamples=24, nburn=3, ngap=2, delta=1e-4, lmda=2e-3, mu=30.0, verbosity=0, complex=False,
                          track=["chain"])
    reg = prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu, L=L, B=B,
                               J_min=J)
    m = mcmc.MYULA(op, reg, p, noise="device", nchains=nch, seed=5, stream0=3)
    m.run(np.random.default_rng(4).laplace(size=(nch, op.nparams)) * 0.05)
    chain = np.asarray(m.chain)
    assert chain.shape == (nch, 24, op.nparams) and not np.iscomplexobj(chain)
    got = px.diag.rank_diagnostics(m.chain)
    check(got, K.rank_diagnostics(chain), "MYULA")


def test_refusals(px):
    torch = px.torch
    rd = px.diag.rank_diagnostics
    with pytest.raises(TypeError):
        rd(np.zeros((2, 8, 3), dtype=complex))
    with pytest.raises(TypeError):
        rd(torch.zeros((2, 8, 3), dtype=torch.complex128, device=px.D.dev()))
    with pytest.raises(ValueError):
        rd(np.zeros((2, 2, 8, 3)))
    with pytest.raises(ValueError, match="16384"):
        rd(np.zeros((5, 3277, 2)))
    with pytest.raises(ValueError, match="16384"):
        rd(torch.zeros((1, 16385, 2), dtype=torch.float64, device=px.D.dev()))
