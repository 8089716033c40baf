"""GPU tests of the streaming posterior summaries (pxm_stats_accumulate / pxm_stats_partials, `summarise=` of the
samplers): the kernels against the two-pass oracle (oracle/diagnostics_ref.py) on seeded device samples, every run loop
against the oracle applied to its own tracked arrays, checkpoint / resume, launch counts and refusals.

Bars (the running moments are Welford / Chan updates, the oracle is two-pass numpy):
  mean            |d| <= 1e-11 (|mu| + lambda) per element
  var, chain_var  1e-10 relative
  R-hat           1e-10 absolute
  ESS, MCSE       1e-9 relative
"""
import numpy as np
import pytest

from oracle import diagnostics_ref as R

pytestmark = pytest.mark.gpu

BARS = {"var": 1e-10, "chain_var": 1e-10, "rhat": 1e-10, "ess": 1e-9, "mcse": 1e-9}


@pytest.fixture(scope="module")
def px():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pxmcmc_b200 import device, diagnostics, forward, mcmc, prior, sht

    class NS:
        pass

    ns = NS()
    ns.D, ns.diag, ns.forward, ns.mcmc, ns.prior, ns.sht = device, diagnostics, forward, mcmc, prior, sht
    return ns


def _nan_same(a, b, what):
    assert np.array_equal(np.isnan(a), np.isnan(b)), what


def check_stats(got, ref, what="", var_bar=None):
    """got: dict of product statistics with trailing shape [ncomp, E] (chain arrays [M, ncomp, E]); ref: oracle dict"""
    lam = np.sqrt(np.abs(ref["var"]))
    lam = np.where(np.isnan(lam), 0.0, lam)
    dm = np.abs(got["mean"] - ref["mean"])
    assert np.all(dm <= 1e-11 * (np.abs(ref["mean"]) + lam) + 1e-300), f"{what} mean: {np.max(dm)}"
    dcm = np.abs(got["chain_mean"] - ref["chain_mean"])
    sc = np.sqrt(np.abs(np.nan_to_num(ref["chain_var"])))
    assert np.all(dcm <= 1e-11 * (np.abs(ref["chain_mean"]) + sc) + 1e-300), f"{what} chain_mean: {np.max(dcm)}"
    for k, bar in BARS.items():
        if var_bar is not None and k in ("var", "chain_var"):
            bar = var_bar
        if var_bar is not None and k not in ("var", "chain_var"):
            continue
        a, b = np.asarray(got[k]), np.asarray(ref[k])
        _nan_same(a, b, f"{what} {k}")
        ok = ~np.isnan(b)
        d = np.abs(a[ok] - b[ok])
        lim = bar if k == "rhat" else bar * np.abs(b[ok])
        assert np.all(d <= lim), f"{what} {k}: worst {np.max(d / np.maximum(lim, 1e-300))} of the bar"


def device_stats(px, acc, n, nch, mode, nsamples):
    """product statistics of an accumulator, in the oracle's layout"""
    rec, cm, cv = px.D.stats_partials_dev(acc, n, nch, mode, nsamples)
    rec = rec.cpu().numpy()
    ncomp = rec.shape[1]
    mean, var, rhat, ess, mcse = px.diag.statistics(rec, nsamples)
    M = cm.shape[0] // ncomp
    return {"mean": mean, "var": var, "rhat": rhat, "ess": ess, "mcse": mcse,
            "chain_mean": cm.cpu().numpy().reshape(M, ncomp, n), "chain_var": cv.cpu().numpy().reshape(M, ncomp, n)}


def logical(xs, mode):
    """host samples [n, nchains, E] complex -> the oracle's [M, n, ncomp, E] real samples of a mode"""
    x = np.moveaxis(np.asarray(xs), 0, 1)  # [nch, n, E]
    if mode == 0:
        return x.real[:, :, None]
    if mode == 1:
        return np.stack([x.real, x.imag], axis=2)
    out = np.empty((2 * x.shape[0],) + x.shape[1:])
    out[0::2], out[1::2] = x.real, x.imag
    return out[:, :, None]


CASES = [(1, 3), (2, 2), (3, 65), (4, 1), (7, 64), (100, 3), (101, 2), (1024, 3), (7, 1), (4, 65)]


@pytest.mark.parametrize("nsamp,nch", CASES)
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_kernel_against_oracle(px, nsamp, nch, mode):
    import torch

    E = 300 if nsamp >= 100 else 517  # not multiples of the block size
    g = torch.Generator(device="cuda").manual_seed(1000 * nsamp + 10 * nch + mode)
    scale = [1e-6, 1.0, 1e6][(nsamp + nch) % 3]
    chain_scale = scale * torch.exp(torch.rand((nch, 1), generator=g, device="cuda", dtype=torch.float64) - 0.5)
    offs = torch.randn((nch, 1), generator=g, device="cuda", dtype=torch.float64) * scale * 0.3
    acc = px.D.stats_accumulator(E, nch, mode)
    acc.fill_(float("nan"))  # handed over dirty: nothing of it may reach a statistic
    px.D.lib.pxm_stats_reset(px.D.ptr(acc), E, nch, mode, px.D.stream_ptr())
    acc2 = px.D.stats_accumulator(E, nch, mode)
    acc2.fill_(float("nan"))  # not even without the reset: every field is overwritten before it is read
    host = []
    for j in range(nsamp):
        x = torch.complex(torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64),
                          torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64)) * chain_scale + offs
        px.D.stats_accumulate_dev(acc, x, mode, nsamp, j=j)
        px.D.stats_accumulate_dev(acc2, x, mode, nsamp, j=j)
        host.append(x.cpu().numpy())
    ref = R.summarise(logical(host, mode))
    got = device_stats(px, acc, E, nch, mode, nsamp)
    check_stats(got, ref, f"n={nsamp} m={nch} mode={mode}")
    got2 = device_stats(px, acc2, E, nch, mode, nsamp)
    for k in got:
        assert np.array_equal(got[k], got2[k], equal_nan=True), k


def test_kernel_per_chain_sample_index(px):
    """d_j: every chain takes its own sample index (PxMALA's accepted samples); -1 skips the chain"""
    import torch

    nch, E, nsamp = 5, 333, 23
    rng = np.random.default_rng(3)
    g = torch.Generator(device="cuda").manual_seed(3)
    acc = px.D.stats_accumulator(E, nch, 1)
    js = np.zeros(nch, dtype=np.int64)
    samples = [[] for _ in range(nch)]
    while js.min() < nsamp:
        x = torch.complex(torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64),
                          torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64))
        take = (rng.uniform(size=nch) < 0.6) & (js < nsamp)
        jd = np.where(take, js, -1)
        px.D.stats_accumulate_dev(acc, x, 1, nsamp, d_j=torch.from_numpy(jd).cuda())
        xh = x.cpu().numpy()
        for c in np.nonzero(take)[0]:
            samples[c].append(xh[c])
        js += take
    xs = np.stack([np.stack(s) for s in samples], axis=1)  # [n, nch, E]
    check_stats(device_stats(px, acc, E, nch, 1, nsamp), R.summarise(logical(xs, 1)), "d_j")


def test_kernel_large_offset(px):
    """mean / std = 1e6: the running (Welford) variance keeps 1e-7; a sum-of-squares formulation loses everything"""
    import torch

    nch, E, nsamp = 4, 1000, 64
    g = torch.Generator(device="cuda").manual_seed(9)
    acc = px.D.stats_accumulator(E, nch, 0)
    host = []
    for j in range(nsamp):
        x = (1e6 + torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64)).to(torch.complex128)
        px.D.stats_accumulate_dev(acc, x, 0, nsamp, j=j)
        host.append(x.cpu().numpy())
    check_stats(device_stats(px, acc, E, nch, 0, nsamp), R.summarise(logical(host, 0)), "offset", var_bar=1e-7)


def test_kernel_bench_shape(px):
    """64 chains x 398 342 coefficients (L = 256, B = 1.5), 5 pushes, checked on a seeded subset of 4 096 elements"""
    import torch

    nch, E, nsamp = 64, 398342, 5
    sub = np.sort(np.random.default_rng(0).choice(E, 4096, replace=False))
    subd = torch.from_numpy(sub).cuda()
    g = torch.Generator(device="cuda").manual_seed(11)
    accs = {m: px.D.stats_accumulator(E, nch, m) for m in (0, 1, 2)}
    host = []
    for j in range(nsamp):
        x = torch.complex(torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64),
                          torch.randn((nch, E), generator=g, device="cuda", dtype=torch.float64))
        for m, a in accs.items():
            px.D.stats_accumulate_dev(a, x, m, nsamp, j=j)
        host.append(x[:, subd].cpu().numpy())
        del x
    for m, a in accs.items():
        got = device_stats(px, a, E, nch, m, nsamp)
        got = {k: v[..., sub] for k, v in got.items()}
        check_stats(got, R.summarise(logical(host, m)), f"bench shape mode {m}")


def test_argument_checks(px):
    import torch

    from pxmcmc_b200._lib import PxmError

    acc = px.D.stats_accumulator(10, 2, 0)
    x = torch.zeros((2, 10), dtype=torch.complex128, device="cuda")
    with pytest.raises(PxmError):
        px.D.stats_accumulate_dev(acc, x, 0, 5, j=5)  # j >= nsamples
    with pytest.raises(PxmError):
        px.D.stats_accumulate_dev(acc, x, 3, 5, j=0)  # bad mode
    with pytest.raises(PxmError):
        px.D.stats_accumulator(10, 2, 7)
    assert px.D.lib.pxm_stats_accumulator_doubles(0, 2, 0) == -1


# ------------------------------------------------------------------ run loops
def _wavelet_case(px, L=16, nch=4, sampler="MYULA", noise="device", form="harm", complex_=False, nsamples=9, nburn=3,
                  ngap=2, summarise=("chain", "predictions"), real_data=False, delta=1e-4, s=1, **kw):
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
                             s=s, complex=complex_, track=["logposterior", "L2", "prior", "chain", "predictions"])
    reg = px.prior.S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, p.lmda * p.mu, L=L, B=B,
                                  J_min=J)
    cls = getattr(px.mcmc, sampler)
    return cls(op, reg, p, noise=noise, nchains=nch, seed=5, stream0=3, summarise=summarise, **kw), op


def _tracked_oracle(m, name):
    arr = np.asarray(m.chain if name == "chain" else m.preds)
    if m.nchains == 1:
        arr = arr[None]
    if np.iscomplexobj(arr):
        return R.summarise(np.stack([arr.real, arr.imag], axis=2))
    return R.summarise(arr[:, :, None])


def _summary_as_oracle(s):
    """diagnostics.Summary -> the oracle's [ncomp, E] / [M, ncomp, E] layout"""
    out = {}
    cplx = np.iscomplexobj(s.mean)
    for k in ("mean", "chain_mean"):
        v = getattr(s, k)
        out[k] = np.stack([v.real, v.imag], axis=-2) if cplx else v[..., None, :]
    for k in ("var", "rhat", "ess", "mcse"):
        v = getattr(s, k)
        out[k] = v if cplx else v[None]
    out["chain_var"] = np.moveaxis(s.chain_var, 0, 1) if cplx else s.chain_var[:, None]
    return out


def _run(m, start, seed=9):
    np.random.seed(seed)
    m.run(start)
    return m


def _check_run(px, make, what, start_shape=None, **kw):
    """the summary of a run against the oracle on its tracked arrays; the tracked arrays bit-identical to a run
    without summarise"""
    a, op = make(px, **kw)
    nch = a.nchains
    start = np.random.default_rng(4).laplace(size=(nch, op.nparams)) * 0.05
    if nch == 1:
        start = start[0]
    _run(a, start)
    b, _ = make(px, summarise=None, **kw)
    _run(b, start)
    for name in ("logPi", "chain", "preds"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), f"{what}: tracked {name} differs with summarise"
    assert b.summary is None
    for t in ("chain", "predictions"):
        check_stats(_summary_as_oracle(a.summary[t]), _tracked_oracle(a, t), f"{what} {t}")
    return a


@pytest.mark.parametrize("form", ["pix", "ring", "harm"])
@pytest.mark.parametrize("noise,graphed", [("device", True), ("device", False), ("host", False)])
def test_myula_run_summary(px, form, noise, graphed):
    def make(px, **kw):
        m, op = _wavelet_case(px, form=form, noise=noise, **kw)
        m.graph_run = graphed
        return m, op

    _check_run(px, make, f"MYULA {form} {noise} graphed={graphed}")


def test_myula_complex_run_summary(px):
    _check_run(px, lambda px, **kw: _wavelet_case(px, complex_=True, nsamples=7, **kw), "MYULA complex")


@pytest.mark.parametrize("noise", ["device", "host"])
def test_real_pairs_run_summary(px, noise):
    a = _check_run(px, lambda px, **kw: _wavelet_case(px, noise=noise, real_data=True, real_pairs=True, **kw), "pairs")
    b, op = _wavelet_case(px, noise=noise, real_data=True)
    start = np.random.default_rng(4).laplace(size=(4, op.nparams)) * 0.05
    _run(b, start)
    for t in ("chain", "predictions"):  # the packed chains equal the unpacked ones to round-off (~1e-12)
        sa, sb = a.summary[t], b.summary[t]
        lam = np.sqrt(sb.var)
        for k in ("mean", "chain_mean"):
            va, vb = getattr(sa, k), getattr(sb, k)
            assert np.all(np.abs(va - vb) <= 1e-10 * (np.abs(vb) + lam)), (t, k)
        for k in ("var", "chain_var", "rhat", "ess", "mcse"):
            va, vb = getattr(sa, k), getattr(sb, k)
            _nan_same(va, vb, k)
            ok = ~np.isnan(vb)
            assert np.all(np.abs(va[ok] - vb[ok]) <= 1e-10 * np.abs(vb[ok]) + 1e-300), (t, k, np.max(np.abs(va[ok] - vb[ok]) / np.abs(vb[ok])))


def test_pxmala_device_run_summary(px):
    """batched device-resident PxMALA: every chain keeps its own count of accepted grid samples"""

    def make(px, summarise=("chain", "predictions")):
        return _wavelet_case(px, L=16, sampler="PxMALA", nsamples=8, nburn=2, ngap=1, delta=1e-3, summarise=summarise)

    a = _check_run(px, make, "PxMALA device")
    assert a._device_resident() and a.nchains == 4
    assert np.any(a.acceptance_trace == 0)  # the chains did reject: per-chain sample indices differ


def test_pxmala_host_loop_run_summary(px):
    def make(px, summarise=("chain", "predictions")):
        return _wavelet_case(px, L=16, nch=1, sampler="PxMALA", noise="host", nsamples=6, nburn=1, ngap=1, delta=1e-5,
                             summarise=summarise)

    a = _check_run(px, make, "PxMALA host")
    assert not a._device_resident()


def test_skrock_run_summary(px):
    def make(px, summarise=("chain", "predictions")):
        return _wavelet_case(px, sampler="SKROCK", nsamples=6, nburn=1, ngap=2, s=3, delta=1e-6, summarise=summarise)

    _check_run(px, make, "SKROCK")


class _Stop(Exception):
    pass


@pytest.mark.parametrize("sampler", ["MYULA", "PxMALA"])
def test_checkpoint_resume_summary_bit_identical(px, sampler, tmp_path):
    """interrupted at an iteration whose sample index lies mid-batch and in the first half (nsamples 20: h = 10,
    b = 4), resumed by a new sampler: the summary is bit for bit the uninterrupted one"""
    kw = dict(sampler=sampler, nsamples=20, nburn=2, ngap=1, L=16)
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
        first.run(start, checkpoint=ck, checkpoint_every=9)  # MYULA: samples j = 0..6 taken, j = 7
    with np.load(ck) as f:
        j = int(f["j"]) if "j" in f.files else int(f["js"].max())
    assert 0 < j < 10 and (sampler != "MYULA" or j % 4 != 0)
    second, _ = _wavelet_case(px, **kw)
    np.random.seed(1234)
    second.run(resume=ck)
    for t in ("chain", "predictions"):
        for k in full.summary[t].STATS:
            assert np.array_equal(getattr(second.summary[t], k), getattr(full.summary[t], k), equal_nan=True), (t, k)
    assert np.array_equal(second.chain, full.chain)
    with pytest.raises(ValueError):  # a checkpoint without accumulators cannot continue a summary
        plain, _ = _wavelet_case(px, summarise=None, **kw)
        plain.run(start, checkpoint=ck)
        _wavelet_case(px, **kw)[0].run(resume=ck)


def test_launch_count(px):
    """one accumulate launch per grid sample and target, nothing off the grid; summarise=None adds nothing"""
    from pxmcmc_b200._lib import lib

    def launches(summarise, ngap, nburn, **kw):
        m, op = _wavelet_case(px, summarise=summarise, ngap=ngap, nburn=nburn, nsamples=5, **kw)
        start = np.random.default_rng(4).laplace(size=(4, op.nparams)) * 0.05
        m.run(start)  # (warm-up: tables, graphs)
        n0 = lib.pxm_launch_count()
        np.random.seed(9)
        m.run(start)
        return lib.pxm_launch_count() - n0

    for ngap, nburn in ((1, 0), (3, 4)):
        base = launches(None, ngap, nburn)
        one = launches(("chain",), ngap, nburn)
        assert one - base == 5 + 1, (ngap, nburn, one - base)  # 5 accumulates + 1 partials at the end
    m, _ = _wavelet_case(px, summarise=None)
    assert m._summarise == ()


def test_refusals(px):
    m, _ = _wavelet_case(px)
    with pytest.raises(NotImplementedError):
        m.iterate_host(np.zeros((4, m.forward.nparams), complex))
    with pytest.raises(ValueError):
        _wavelet_case(px, summarise=("chain", "logposterior"))

    m2, op = _wavelet_case(px, summarise=None)
    op._pxm_allreduce = lambda t: t  # what an m-sharded operator carries
    with pytest.raises(NotImplementedError, match="m-sharded"):
        px.mcmc.MYULA(op, m2.prior, px.mcmc.PxMCMCParams(nsamples=1, verbosity=0), noise="device", nchains=4,
                      summarise=("chain",))
