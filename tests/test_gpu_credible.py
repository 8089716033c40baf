"""GPU tests of the streaming credible intervals (pxm_credible_push / pxm_credible_finalize, `credible=` of the
samplers).  Every comparison is bit for bit (np.array_equal): the tail heaps keep the very order statistics np.quantile
reads, and the interpolation is numpy's _lerp."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def px():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pxmcmc_b200 import device, diagnostics, forward, mcmc, prior, saving, sht, uncertainty

    class NS:
        pass

    ns = NS()
    ns.D, ns.diag, ns.forward, ns.mcmc, ns.prior, ns.saving, ns.sht, ns.U = (device, diagnostics, forward, mcmc, prior,
                                                                             saving, sht, uncertainty)
    return ns


def _quantiles(pooled, alpha):
    """numpy's (lower, upper) over axis 0"""
    with np.errstate(invalid="ignore"):
        return np.quantile(pooled, alpha / 2, axis=0), np.quantile(pooled, 1 - alpha / 2, axis=0)


def _pooled(samples, mode):
    """host samples: list of complex [nchains, E] pushes, each restricted to the chains that took a sample ->
    [N, E] (modes 0, 2) or [N, 2, E] (mode 1) pooled logical values"""
    x = np.concatenate(samples, axis=0)
    if mode == 0:
        return x.real
    if mode == 1:
        return np.stack([x.real, x.imag], axis=1)
    return np.concatenate([x.real, x.imag], axis=0)


def _device(px, mode, alpha, pushes, E, d_js=None):
    """push [nchains, E] complex device tensors (with per-push d_j int64 host arrays) -> (lower, upper) host arrays"""
    import torch

    nch = pushes[0].shape[0]
    parts = 2 if mode == 2 else 1
    active = [nch if d_js is None else int((d >= 0).sum()) for d in (d_js or [None] * len(pushes))]
    tails = px.diag.credible_tails(sum(active) * parts, alpha)
    st = px.D.credible_state(E, mode, tails)
    count = 0
    for k, x in enumerate(pushes):
        dj = None if d_js is None else torch.from_numpy(d_js[k]).cuda()
        px.D.credible_push_dev(st, x, mode, tails, count, dj)
        count += active[k] * parts
    lo, hi = px.D.credible_finalize_dev(st, E, mode, tails)
    lo, hi = lo.cpu().numpy(), hi.cpu().numpy()
    return (lo, hi) if mode == 1 else (lo[0], hi[0])


def _data(rng, nch, E):
    """complex [nch, E]: per column group iid normal, heavy ties, signed zeros, Cauchy, +-inf, rare NaN"""
    def part():
        v = rng.standard_normal((nch, E))
        k = np.arange(E) % 6
        v[:, k == 1] = np.floor(v[:, k == 1] * 2)
        z = rng.uniform(size=(nch, E)) < 0.6
        v[:, k == 2] = np.where(z, np.where(rng.uniform(size=(nch, E)) < 0.5, 0.0, -0.0), v)[:, k == 2]
        v[:, k == 3] = rng.standard_cauchy((nch, int((k == 3).sum())))
        u = rng.uniform(size=(nch, E))
        v[:, k == 4] = np.where(u < 0.05, np.inf, np.where(u > 0.95, -np.inf, v))[:, k == 4]
        v[:, k == 5] = np.where(u < 0.003, np.nan, v)[:, k == 5]
        return v
    x = np.empty((nch, E), dtype=np.complex128)  # (not re + 1j * im: 1j * inf has a NaN real part)
    x.real, x.imag = part(), part()
    return x


SHAPES = [(1, 1), (1, 257), (2, 3), (3, 2), (3, 7), (2, 40), (64, 2), (64, 7)]


@pytest.mark.parametrize("nch,nsamp", SHAPES)
@pytest.mark.parametrize("alpha", [0.001, 0.05, 0.1, 0.5, 0.9])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_kernel_against_numpy(px, nch, nsamp, alpha, mode):
    import torch

    E = 517  # not a multiple of the block
    rng = np.random.default_rng(1000 * nsamp + 10 * nch + mode + int(alpha * 1000))
    host = [_data(rng, nch, E) for _ in range(nsamp)]
    lo, hi = _device(px, mode, alpha, [torch.from_numpy(x).cuda() for x in host], E)
    rlo, rhi = _quantiles(_pooled(host, mode), alpha)
    assert np.array_equal(lo, rlo, equal_nan=True) and np.array_equal(hi, rhi, equal_nan=True)
    assert not np.isnan(lo[..., np.arange(E) % 6 == 0]).any()


def test_reference_golden_vectors(px):
    """the chains of tests/golden/ref_uncertainty.npz (37 to 5 000 samples), one sample per push: the range is the
    unmodified reference's credible_interval_range, and the wavelet split its wavelet_credible_interval_range"""
    import torch
    from conftest import golden

    from oracle.gen_golden_uncertainty import CASES, make_chain

    g = golden("ref_uncertainty.npz")
    for i, (n, p, seed) in enumerate(CASES):
        x = torch.from_numpy(make_chain(n, p, seed)).to(torch.complex128).cuda()
        for alpha, key in ((0.05, f"ci_{i}"), (0.1, f"ci10_{i}")):
            lo, hi = _device(px, 0, alpha, [x[j:j + 1] for j in range(n)], p)
            ci = px.diag.CredibleIntervals(alpha, 1, n, lo, hi)
            assert np.array_equal(ci.range, g[key]), key
            if i == 0 and alpha == 0.05:
                maps = ci.wavelet_maps("range", 10, 2, 2)
                assert [list(m.shape) for m in maps] == g["wav_shapes"].tolist()
                assert np.array_equal(np.concatenate([m.ravel() for m in maps]), g["wav_flat"])


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_per_chain_sample_indices(px, mode):
    """d_j with -1 entries before, across and after the fill boundary: exactly the pushed samples count"""
    import torch

    nch, E, alpha = 5, 333, 0.3
    rng = np.random.default_rng(3 + mode)
    pushes, d_js, taken = [], [], []
    for k in range(30):
        x = _data(rng, nch, E)
        take = rng.uniform(size=nch) < 0.5
        if k == 0:
            take[:] = False
        d_js.append(np.where(take, k, -1).astype(np.int64))
        pushes.append(torch.from_numpy(x).cuda())
        taken.append(x[take])
    lo, hi = _device(px, mode, alpha, pushes, E, d_js)
    rlo, rhi = _quantiles(_pooled(taken, mode), alpha)
    assert np.array_equal(lo, rlo, equal_nan=True) and np.array_equal(hi, rhi, equal_nan=True)


def test_order_independence(px):
    """the same 96 values per column as 4 chains x 24 pushes, 24 chains x 4 pushes in permuted order and 1 chain x 96
    pushes: bit-identical intervals"""
    import torch

    E, alpha = 700, 0.1
    rng = np.random.default_rng(17)
    vals = _data(rng, 96, E)
    a = [torch.from_numpy(vals[4 * k:4 * k + 4]).cuda() for k in range(24)]
    perm = vals[rng.permutation(96)]
    b = [torch.from_numpy(perm[24 * k:24 * k + 24]).cuda() for k in range(4)]
    c = [torch.from_numpy(vals[k:k + 1]).cuda() for k in rng.permutation(96)]
    ra, rb, rc = (_device(px, 0, alpha, s, E) for s in (a, b, c))
    for x in (rb, rc):
        assert np.array_equal(ra[0], x[0], equal_nan=True) and np.array_equal(ra[1], x[1], equal_nan=True)
    rlo, rhi = _quantiles(vals.real, alpha)
    assert np.array_equal(ra[0], rlo, equal_nan=True) and np.array_equal(ra[1], rhi, equal_nan=True)


def _subset_run(px, nch, E, nsamp, alpha, modes, seed, sub):
    """device-generated pushes of nch x E, every mode in `modes` fed the same samples; host copies of columns `sub`"""
    import torch

    subd = torch.from_numpy(sub).cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    parts = {m: 2 if m == 2 else 1 for m in modes}
    tails = {m: px.diag.credible_tails(nch * nsamp * parts[m], alpha) for m in modes}
    st = {m: px.D.credible_state(E, m, tails[m]) for m in modes}
    host = []
    for j in range(nsamp):
        x = torch.complex(torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64),
                          torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64))
        for m in modes:
            px.D.credible_push_dev(st[m], x, m, tails[m], j * nch * parts[m])
        host.append(x[:, subd].cpu().numpy())
        del x
    for m in modes:
        lo, hi = px.D.credible_finalize_dev(st[m], E, m, tails[m])
        del st[m]
        lo, hi = lo.cpu().numpy()[..., sub], hi.cpu().numpy()[..., sub]
        if m != 1:
            lo, hi = lo[0], hi[0]
        rlo, rhi = _quantiles(_pooled(host, m), alpha)
        assert np.array_equal(lo, rlo) and np.array_equal(hi, rhi), m


def test_bench_shape(px):
    """64 chains x 398 342 coefficients (L = 256, B = 1.5), 40 samples per chain, on a seeded subset of 4 096"""
    E = 398342
    sub = np.sort(np.random.default_rng(0).choice(E, 4096, replace=False))
    _subset_run(px, 64, E, 40, 0.05, (0, 1, 2), 11, sub)


def test_heap_index_past_2_31(px):
    """one chain, 4.2 M elements, alpha = 0.9, 1 200 samples: K = 541 per tail, heap offsets up to 2.3e9 doubles"""
    import torch

    E, nsamp, alpha = 4_200_000, 1200, 0.9
    _, lo_a, _, lo_b, _ = px.diag.credible_tails(nsamp, alpha)
    assert min(lo_a + 2, nsamp) == 541 and nsamp - lo_b == 541
    if torch.cuda.mem_get_info()[0] < 40e9:
        pytest.skip("needs 40 GB of free device memory")
    sub = np.sort(np.concatenate([np.random.default_rng(1).choice(E, 4090, replace=False), [0, 1, E - 2, E - 1]]))
    sub = np.unique(sub)
    _subset_run(px, 1, E, nsamp, alpha, (0,), 5, sub)


def test_argument_checks(px):
    import torch

    from pxmcmc_b200._lib import PxmError

    lib = px.D.lib
    assert lib.pxm_credible_state_doubles(0, 0, 10, 1, 8) == -1
    assert lib.pxm_credible_state_doubles(10, 3, 10, 1, 8) == -1
    assert lib.pxm_credible_state_doubles(10, 0, 10, 10, 8) == -1
    assert lib.pxm_credible_state_doubles(10, 0, 0, 0, 0) == -1
    assert lib.pxm_credible_state_doubles(10, 1, 10, 1, 8) == (3 + 2 + 1) * 20
    tails = px.diag.credible_tails(4, 0.5)
    st = px.D.credible_state(10, 0, tails)
    x = torch.zeros((2, 10), dtype=torch.complex128, device="cuda")
    with pytest.raises(PxmError):
        px.D.credible_push_dev(st, x, 0, tails, 5)  # count > npooled
    with pytest.raises(PxmError):
        px.D.credible_push_dev(st, x, 3, tails, 0)  # bad mode


# ------------------------------------------------------------------ samplers
def _wavelet_case(px, L=16, nch=4, sampler="MYULA", noise="device", form="harm", complex_=False, nsamples=9, nburn=3,
                  ngap=2, credible=("chain", "predictions"), alpha=0.2, real_data=False, delta=1e-4, s=1,
                  summarise=("chain",), track=("logposterior", "L2", "prior", "chain", "predictions"), **kw):
    B, J = 1.5, 2
    rng = np.random.default_rng(12)
    flm = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    data = px.sht.inverse(flm, L).ravel()
    if real_data:
        data = np.ascontiguousarray(data.real)
    op = px.forward.SphericalWaveletTransformOperator(data, 0.3, "synthesis", L, B, J, nchains=nch)
    op.fuse_ring = form in ("ring", "harm")
    op.fuse_gram = form == "harm"
    p = px.mcmc.PxMCMCParams(nsamples=nsamples, nburn=nburn, ngap=ngap, delta=delta, lmda=2e-3, mu=30.0, verbosity=0,
                             s=s, complex=complex_, track=list(track))
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu, L=L, B=B,
                                  J_min=J)
    cls = getattr(px.mcmc, sampler)
    return cls(op, reg, p, noise=noise, nchains=nch, seed=5, stream0=3, summarise=summarise, credible=credible,
               credible_alpha=alpha, **kw), op


def _run(m, start, seed=9):
    np.random.seed(seed)
    m.run(start)
    return m


def _tracked_quantiles(m, name, alpha):
    arr = np.asarray(m.chain if name == "chain" else m.preds)
    E = arr.shape[-1]
    if np.iscomplexobj(arr) and name == "chain" and m.complex:
        flat = arr.reshape(-1, E)
        return _quantiles(np.stack([flat.real, flat.imag], axis=1), alpha)
    return _quantiles(arr.real.reshape(-1, E), alpha)


def _check_run(px, make, what):
    """the intervals of a run against np.quantile over its own tracked arrays; tracked arrays and summaries
    bit-identical to a run without credible"""
    a, op = make(px)
    nch = a.nchains
    start = np.random.default_rng(4).laplace(size=(nch, op.nparams)) * 0.05
    if nch == 1:
        start = start[0]
    _run(a, start)
    b, _ = make(px, credible=None)
    _run(b, start)
    for name in ("logPi", "chain", "preds"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), f"{what}: tracked {name} differs with credible"
    for k in b.summary["chain"].STATS:
        assert np.array_equal(getattr(a.summary["chain"], k), getattr(b.summary["chain"], k), equal_nan=True), k
    assert b.credible_intervals is None
    for t in ("chain", "predictions"):
        ci = a.credible_intervals[t]
        rlo, rhi = _tracked_quantiles(a, t, ci.alpha)
        assert np.array_equal(ci.lower, rlo) and np.array_equal(ci.upper, rhi), f"{what} {t}"
        assert np.array_equal(ci.range, rhi - rlo)
        assert ci.npooled == ci.nchains * ci.nsamples == np.asarray(a.chain).reshape(-1, op.nparams).shape[0]
    if nch == 1:
        assert np.array_equal(a.credible_intervals["chain"].range,
                              px.U.credible_interval_range(np.asarray(a.chain).real, a.credible_intervals["chain"].alpha))
    return a


@pytest.mark.parametrize("form", ["pix", "ring", "harm"])
@pytest.mark.parametrize("noise,graphed", [("device", True), ("device", False), ("host", False)])
def test_myula_run(px, form, noise, graphed):
    def make(px, **kw):
        m, op = _wavelet_case(px, form=form, noise=noise, **kw)
        m.graph_run = graphed
        return m, op

    _check_run(px, make, f"MYULA {form} {noise} graphed={graphed}")


def test_myula_complex_run(px):
    a = _check_run(px, lambda px, **kw: _wavelet_case(px, complex_=True, nsamples=7, **kw), "MYULA complex")
    assert a.credible_intervals["chain"].lower.shape == (2, a.forward.nparams)


@pytest.mark.parametrize("noise", ["device", "host"])
def test_real_pairs_run(px, noise):
    a = _check_run(px, lambda px, **kw: _wavelet_case(px, noise=noise, real_data=True, real_pairs=True, **kw), "pairs")
    assert a.credible_intervals["chain"].nchains == 4


def test_pxmala_device_run(px):
    def make(px, credible=("chain", "predictions")):
        return _wavelet_case(px, L=16, sampler="PxMALA", nsamples=8, nburn=2, ngap=1, delta=1e-3, credible=credible)

    a = _check_run(px, make, "PxMALA device")
    assert a._device_resident() and a.nchains == 4
    assert np.any(a.acceptance_trace == 0)  # the chains did reject: per-chain sample indices differ


def test_pxmala_host_loop_run(px):
    def make(px, credible=("chain", "predictions")):
        return _wavelet_case(px, L=16, nch=1, sampler="PxMALA", noise="host", nsamples=6, nburn=1, ngap=1, delta=1e-5,
                             credible=credible)

    a = _check_run(px, make, "PxMALA host")
    assert not a._device_resident()


def test_skrock_run(px):
    def make(px, credible=("chain", "predictions")):
        return _wavelet_case(px, sampler="SKROCK", nsamples=6, nburn=1, ngap=2, s=3, delta=1e-6, credible=credible)

    _check_run(px, make, "SKROCK")


class _Stop(Exception):
    pass


@pytest.mark.parametrize("sampler", ["MYULA", "PxMALA"])
@pytest.mark.parametrize("every", [4, 15])
def test_checkpoint_resume_bit_identical(px, sampler, every, tmp_path):
    """4 chains x 20 samples at alpha = 0.5 (K_lo = 21 of N = 80): interrupted while the heaps fill (every = 4) and
    after (every = 15), resumed by a new sampler: bit-identical intervals"""
    kw = dict(sampler=sampler, nsamples=20, nburn=2, ngap=1, L=16, alpha=0.5, summarise=None)
    start = np.random.default_rng(4).laplace(size=(4, _wavelet_case(px, **kw)[1].nparams)) * 0.05
    full, _ = _wavelet_case(px, **kw)
    _run(full, start)
    first, _ = _wavelet_case(px, **kw)
    ck = str(tmp_path / "ck.npz")
    orig = first._save_ckpt

    def save_then_stop(path, **f):
        orig(path, **f)
        raise _Stop

    first._save_ckpt = save_then_stop
    with pytest.raises(_Stop):
        np.random.seed(9)
        first.run(start, checkpoint=ck, checkpoint_every=every)
    with np.load(ck) as f:
        count = int(f["cred_count"])
    assert 0 < count < 21 if every == 4 else count > 21
    second, _ = _wavelet_case(px, **kw)
    np.random.seed(1234)
    second.run(resume=ck)
    for t in ("chain", "predictions"):
        a, b = second.credible_intervals[t], full.credible_intervals[t]
        assert np.array_equal(a.lower, b.lower) and np.array_equal(a.upper, b.upper), t
    assert np.array_equal(second.chain, full.chain)
    assert not any(k.startswith("cred_") for k in second._load_ckpt(ck))
    with pytest.raises(ValueError, match="credible"):  # a checkpoint without heaps cannot continue the intervals
        plain, _ = _wavelet_case(px, **dict(kw, credible=None))
        plain.run(start, checkpoint=ck)
        _wavelet_case(px, **kw)[0].run(resume=ck)


def test_launch_count(px):
    """one push per grid sample and target, one finalize per target; credible=None adds nothing"""
    from pxmcmc_b200._lib import lib

    def launches(credible, ngap, nburn, form="harm"):
        m, op = _wavelet_case(px, credible=credible, summarise=None, ngap=ngap, nburn=nburn, nsamples=5, form=form)
        start = np.random.default_rng(4).laplace(size=(4, op.nparams)) * 0.05
        m.run(start)  # (warm-up: tables, graphs)
        n0 = lib.pxm_launch_count()
        np.random.seed(9)
        m.run(start)
        return lib.pxm_launch_count() - n0

    for ngap, nburn in ((1, 0), (3, 4)):
        base = launches(None, ngap, nburn)
        assert launches(("chain",), ngap, nburn) - base == 5 + 1
        # (pixel form: predictions in ring or Gram form are converted to pixels for tracking in any case)
        pix = launches(None, ngap, nburn, "pix")
        assert launches(("chain", "predictions"), ngap, nburn, "pix") - pix == 2 * (5 + 1)
    m, _ = _wavelet_case(px, credible=None)
    assert m._credible == () and m._cred is None and m.credible_intervals is None


def test_refusals(px):
    for alpha in (0.0, 1.0, 1.5, -0.1, float("nan")):
        with pytest.raises(ValueError, match="credible_alpha"):
            _wavelet_case(px, alpha=alpha)
    with pytest.raises(ValueError):
        _wavelet_case(px, credible=("chain", "logposterior"))
    with pytest.raises(ValueError):
        _wavelet_case(px, credible=())
    m, _ = _wavelet_case(px, summarise=None)
    with pytest.raises(NotImplementedError):
        m.iterate_host(np.zeros((4, m.forward.nparams), complex))
    m2, op = _wavelet_case(px, credible=None, summarise=None)
    op._pxm_allreduce = lambda t: t  # what an m-sharded operator carries
    with pytest.raises(NotImplementedError, match="m-sharded"):
        px.mcmc.MYULA(op, m2.prior, px.mcmc.PxMCMCParams(nsamples=1, verbosity=0), noise="device", nchains=4,
                      credible=("chain",))
    big, op = _wavelet_case(px, nsamples=10 ** 9, alpha=0.9, summarise=None, track=())
    with pytest.raises(ValueError, match="bytes"):  # sized at run start: more than the device holds
        big.run(np.zeros((4, op.nparams)))


def test_saving_round_trip(px, tmp_path):
    m, op = _wavelet_case(px, nsamples=5)
    _run(m, np.random.default_rng(4).laplace(size=(4, op.nparams)) * 0.05)
    p = px.mcmc.PxMCMCParams(nsamples=5, verbosity=0)
    path = px.saving.save_mcmc(m, p, str(tmp_path), "with")
    data, _ = px.saving.load_mcmc(path)
    got = px.saving.credible_intervals(data)
    assert sorted(got) == ["chain", "predictions"]
    for t, ci in m.credible_intervals.items():
        g = got[t]
        assert (g.alpha, g.nchains, g.nsamples) == (ci.alpha, ci.nchains, ci.nsamples)
        for k in ("lower", "upper", "range"):
            assert np.array_equal(getattr(g, k), getattr(ci, k)), (t, k)
    assert sorted(px.saving.summaries(data)) == ["chain"]
    plain, _ = _wavelet_case(px, nsamples=5, credible=None)
    _run(plain, np.random.default_rng(4).laplace(size=(4, op.nparams)) * 0.05)
    data2, _ = px.saving.load_mcmc(px.saving.save_mcmc(plain, p, str(tmp_path), "without"))
    assert not any(k.startswith("credible/") for k in data2) and px.saving.credible_intervals(data2) == {}
    assert sorted(data2) == sorted(k for k in data if not k.startswith("credible/"))
