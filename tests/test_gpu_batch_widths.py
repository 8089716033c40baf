"""GPU parity at the batch widths the samplers run (`pytest -m gpu`).

The bench's MYULA step runs 64 chains per GPU.  The width decides which kernels run: a wavelet plan of `nb` chains has
nld = pad(4 nb) Legendre columns (pad: 8, 16, 32, 64, then multiples of 128), the contraction runs the BN = nld
instantiation below 128 columns and BN = 128 with nld / 128 column blocks above (whose producer copies one row group at
a time, at stride nld), and the ring FFT picks the persistent TMA-staged kernel once the grid has 700 CTAs or more.
Every chain is compared with the CPU oracle on its own, so a small chain cannot hide behind a large one.

The oracle cost stays fixed with linearity: chain c of a batch is x_c = sum_k a_ck u_k over K basis inputs, with chain
scales spread over 1e-6 ... 1, and its expected output is sum_k a_ck T(u_k) with T(u_k) from the oracle.  The noise of
the Philox kernels is compared with the host restatement in oracle/philox_ref.py.
"""
import os
from concurrent.futures import ProcessPoolExecutor
import multiprocessing as mp

import numpy as np
import pytest
from scipy import sparse

from conftest import rel_l2
from oracle import philox_ref

pytestmark = pytest.mark.gpu

TOL = 1e-10
K = 3

# transform width sweep: Bluestein lengths of the <= 256, 512 and 1024 classes; nld 8 ... 384
LW, BW, JW = 130, 2.0, 2
WIDTHS = [1, 2, 3, 5, 8, 9, 16, 17, 32, 33, 64, 65]
CALLS = [(w, w) for w in WIDTHS] + [(65, 1), (65, 33), (65, 64)]  # (plan width, chains in the call)
IC = 0.7 - 0.3j  # inverse covariance of the Gram-form gradient


# ------------------------------------------------------------------ oracle workers (CPU processes)
def _limit_threads():
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=1)
    except Exception:  # noqa: BLE001
        pass


def _w_oracle(args):
    name, x, L, B, J = args
    _limit_threads()
    from oracle import pxmcmc_ref as R
    from oracle import ssht_ref

    if name.startswith("sht"):
        spin, fn = int(name[3]), name[5:]
        if fn in ("forward", "inverse_adjoint"):
            x = x.reshape(L, 2 * L - 1)
        return np.asarray(getattr(ssht_ref, fn)(x, L, spin)).ravel()
    t = R.WaveletTransform(L, B, J)
    if name == "harmonic":  # coefficients -> f_lm of the image (the synthesis is band-limited: the forward SHT is exact)
        return np.asarray(ssht_ref.forward(t.inverse(x).reshape(L, 2 * L - 1), L, 0)).ravel()
    if name == "harmonic_adjoint":
        return t.inverse_adjoint(np.asarray(ssht_ref.forward_adjoint(x, L, 0)).ravel())
    if name == "normal":  # Psi^dagger Psi
        return t.inverse_adjoint(t.inverse(x))
    if name.startswith("normal_w"):  # Psi^dagger (ic Psi), x = (u, ic)
        return t.inverse_adjoint(x[1] * t.inverse(x[0]))
    return getattr(t, name)(x)


@pytest.fixture(scope="module")
def pool():
    n = max(1, min(8, (os.cpu_count() or 2) - 1))
    with ProcessPoolExecutor(n, mp_context=mp.get_context("spawn")) as ex:
        yield ex


@pytest.fixture(scope="module")
def torch_dev():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def chain_coefficients(nb, seed, real=False):
    """a [nb, K]: random (complex) directions, chain scales 1 ... 1e-6 in shuffled order"""
    rng = np.random.default_rng(seed)
    scales = rng.permutation(np.logspace(0, -6, nb))
    a = rng.standard_normal((nb, K)) if real else _crandn(rng, nb, K)
    return a * scales[:, None]


# ------------------------------------------------------------------ (a) transform width sweep
# name -> (input kind, oracle operation)
OPS = {
    "synthesis": ("coef", "inverse"),
    "synthesis_adjoint": ("pix", "inverse_adjoint"),
    "analysis": ("pix", "forward"),
    "analysis_adjoint": ("coef", "forward_adjoint"),
    "synthesis_harmonic": ("coef", "harmonic"),
    "synthesis_adjoint_harmonic": ("flm0", "harmonic_adjoint"),
    "synthesis_to_ring+ring_to_pix": ("coef", "inverse"),
    "synthesis_to_harm+harm_to_pix": ("coef", "inverse"),
    "synthesis_to_harm+gram_gradient": ("coef", "normal"),
}
for _s in (0, 2):
    OPS.update({f"sht{_s}_inverse": (f"flm{_s}", f"sht{_s}_inverse"), f"sht{_s}_forward": ("pix", f"sht{_s}_forward"),
                f"sht{_s}_inverse_adjoint": ("pix", f"sht{_s}_inverse_adjoint"),
                f"sht{_s}_forward_adjoint": (f"flm{_s}", f"sht{_s}_forward_adjoint")})
WAVELET_OPS = ("synthesis", "synthesis_adjoint", "analysis", "analysis_adjoint")


@pytest.fixture(scope="module")
def sweep_oracle(pool):
    """basis inputs u_k of every input kind, T(u_k) of every operation, and the data term of the Gram gradient"""
    L = LW
    rng = np.random.default_rng(130)
    from oracle import pxmcmc_ref as R

    ncoefs = R.WaveletTransform(LW, BW, JW).ncoefs
    U = {"coef": _crandn(rng, K, ncoefs), "pix": _crandn(rng, K, L * (2 * L - 1)), "flm0": _crandn(rng, K, L * L),
         "flm2": _crandn(rng, K, L * L)}
    U["flm2"][:, :4] = 0
    d = 1e-8 * _crandn(rng, L * (2 * L - 1))  # small: the data term does not swamp the 1e-6 chains
    jobs = [(op, U[kind][k], LW, BW, JW) for kind, op in sorted(set(OPS.values())) for k in range(K)]
    jobs.append(("inverse_adjoint", d, LW, BW, JW))
    res = list(pool.map(_w_oracle, jobs))
    T = {}
    for job, r in zip(jobs[:-1], res[:-1]):
        T.setdefault(job[0], []).append(r)
    T = {op: np.stack(v) for op, v in T.items()}
    T["normal"] = IC * T["normal"]
    offset = {"normal": -IC * res[-1]}
    return U, T, offset, d


def _nan(torch, n):
    return torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")


def _poison_allocator(torch, nbytes):
    """fill the caching allocator's free blocks with NaN, so that an output a kernel leaves partly unwritten shows"""
    torch.cuda.synchronize()
    blocks = [torch.full((nbytes // 8,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(4)]
    blocks += [torch.full((1 << s,), float("nan"), dtype=torch.float64, device="cuda") for s in range(8, 17) for _ in range(8)]
    del blocks
    probe = torch.empty(nbytes // 16, dtype=torch.complex128, device="cuda")
    assert bool(torch.isnan(probe.real).all()), "the NaN poison did not reach the allocator's free blocks"
    del probe


def _run_ops(torch, width, nb, X, d):
    """every operation of OPS on the device inputs X[kind] ([nb, n]); host arrays [nb, n_out]"""
    from pxmcmc_b200 import device as D

    wp = D.WaveletPlan.get(LW, BW, JW, width)
    sp = {s: D.ShtPlan.get(LW, s, width) for s in (0, 2)}
    wp.set_gram_weights(None)
    b = wp.pix_to_harm_adjoint(D.to_dev_c(d).reshape(1, -1))
    calls = {
        "synthesis": wp.synthesis, "synthesis_adjoint": wp.synthesis_adjoint, "analysis": wp.analysis,
        "analysis_adjoint": wp.analysis_adjoint, "synthesis_harmonic": wp.synthesis_harmonic,
        "synthesis_adjoint_harmonic": wp.synthesis_adjoint_harmonic,
        # carried forms; the ring / harmonic buffers are handed over full of NaN: the kernels must write all of them
        "synthesis_to_ring+ring_to_pix": lambda x: wp.ring_to_pix(wp.synthesis_to_ring(x, out=_nan(torch, wp.ring_doubles)), nb),
        "synthesis_to_harm+harm_to_pix": lambda x: wp.harm_to_pix(wp.synthesis_to_harm(x, out=_nan(torch, wp.harm_doubles)), nb),
        "synthesis_to_harm+gram_gradient": lambda x: wp.gram_gradient(wp.synthesis_to_harm(x, out=_nan(torch, wp.harm_doubles)), b, IC, nb),
    }
    for s in (0, 2):
        for fn in ("inverse", "forward", "inverse_adjoint", "forward_adjoint"):
            calls[f"sht{s}_{fn}"] = getattr(sp[s], fn)
    _poison_allocator(torch, 16 * nb * max(x.shape[1] for x in X.values()))
    out = {name: D.to_host(calls[name](X[OPS[name][0]])) for name in OPS}
    torch.cuda.synchronize()
    return out


def _with_debug(fn, *, fft=None, naive=None):
    from pxmcmc_b200 import _lib

    try:
        if fft is not None:
            _lib.check(_lib.lib.pxm_debug_set_fft_multipass(fft))
        if naive is not None:
            _lib.check(_lib.lib.pxm_debug_set_naive(naive))
        return fn()
    finally:
        _lib.check(_lib.lib.pxm_debug_set_fft_multipass(0))
        _lib.check(_lib.lib.pxm_debug_set_naive(0))


@pytest.mark.parametrize("width,nb", CALLS)
def test_transforms_per_chain_against_oracle(torch_dev, sweep_oracle, width, nb):
    """all four wavelet operators, the harmonic pair, the carried forms and spin-0 / spin-2 SHTs at every Legendre width
    (every BN, both copy branches of the producer, padded columns, an odd number of column blocks), calls narrower than
    the plan included; rel-L2 < 1e-10 per chain"""
    torch = torch_dev
    from pxmcmc_b200 import device as D

    U, T, offset, d = sweep_oracle
    a = chain_coefficients(nb, 1000 * width + nb)
    X = {kind: D.to_dev_c(a @ u) for kind, u in U.items()}
    got = _run_ops(torch, width, nb, X, d)
    wide = nb == width and width >= 33  # nld >= 256: two or three column blocks of BN = 128
    naive = _with_debug(lambda: _run_ops(torch, width, nb, X, d), naive=1) if wide else None
    # the automatic ring-FFT choice: persistent staged kernel at the bench width, multi-pass kernel for one chain
    if nb == width and width in (64, 65):
        forced = _with_debug(lambda: {n: D.to_host(getattr(D.WaveletPlan.get(LW, BW, JW, width), n)(X[OPS[n][0]]))
                                      for n in WAVELET_OPS}, fft=3)
        for n in WAVELET_OPS:
            assert np.array_equal(got[n], forced[n]), f"{n}: default ring FFT at {nb} chains is not the persistent kernel"
    if nb == 1:
        forced = _with_debug(lambda: {n: D.to_host(getattr(D.WaveletPlan.get(LW, BW, JW, width), n)(X[OPS[n][0]]))
                                      for n in WAVELET_OPS}, fft=1)
        for n in WAVELET_OPS:
            assert np.array_equal(got[n], forced[n]), f"{n}: default ring FFT of one chain is not the multi-pass kernel"
    for name, (kind, op) in OPS.items():
        exp = a @ T[op] + offset.get(op, 0)
        assert got[name].shape == exp.shape, name
        for c in range(nb):
            err = rel_l2(got[name][c], exp[c])
            hint = "" if naive is None else f" (plain contraction kernel: {rel_l2(naive[name][c], exp[c]):.2e})"
            assert err < TOL, f"{name}, plan {width}, {nb} chains, chain {c} (scale {np.abs(a[c]).max():.0e}): rel-L2 {err:.2e}{hint}"
            if naive is not None:
                assert rel_l2(got[name][c], naive[name][c]) < 1e-13, f"{name} chain {c}: tensor-core vs plain contraction"


# ------------------------------------------------------------------ (b) the bench step at its real width
LB, BB, JB, NB = 256, 1.5, 2, 64
DELTA = LMDA = 1e-6
SEED = 1234


def _bench_data(real):
    """bench.py's data: A_inv(L, 0) of the synthetic flm, unit RMS, complex (or its real part, unit RMS)"""
    from test_gpu_configs import synthetic_flm

    from oracle import ssht_ref

    d = np.asarray(ssht_ref.inverse(synthetic_flm(LB), LB, 0)).ravel()
    d = d / np.sqrt(np.mean(np.abs(d) ** 2))
    if real:
        d = np.ascontiguousarray(d.real)
        d = d / np.sqrt(np.mean(d ** 2))
    return d


def _ring_sigma():
    return np.repeat(0.5 + np.random.default_rng(5).random(LB), 2 * LB - 1)


MODELS = {  # name -> (sigma, real data, fuse the ring / Gram forms)
    "scalar-gram": (1.0, False, True),
    "per-ring-gram": ("ring", False, True),
    "literal": (1.0, False, False),
    "real-pairs": (1.0, True, True),
}


@pytest.fixture(scope="module")
def bench_oracle(pool):
    """basis states u_k (real), Psi u_k, and per noise model Psi^dagger(ic Psi u_k) and Psi^dagger(ic d)"""
    from oracle import pxmcmc_ref as R

    ncoefs = R.WaveletTransform(LB, BB, JB).ncoefs
    rng = np.random.default_rng(256)
    U = rng.laplace(size=(K, ncoefs)).astype(complex)
    ics = {}
    for name, (sig, real, _) in MODELS.items():
        d = _bench_data(real)
        ics[name] = (d, R.inverse_covariance(d, _ring_sigma() if sig == "ring" else sig))
    jobs = [("inverse", U[k], LB, BB, JB) for k in range(K)]
    for name, (d, ic) in ics.items():
        jobs += [("normal_w", (U[k], ic), LB, BB, JB) for k in range(K)]
        jobs.append(("inverse_adjoint", ic * d, LB, BB, JB))
    res = list(pool.map(_w_oracle, jobs))
    out = {"U": U, "PsiU": np.stack(res[:K])}
    for i, (name, (d, ic)) in enumerate(ics.items()):
        r = res[K + i * (K + 1): K + (i + 1) * (K + 1)]
        out[name] = (d, ic, np.stack(r[:K]), r[K])
    return out


@pytest.mark.parametrize("stream0", [0, 64])
@pytest.mark.parametrize("model", list(MODELS))
def test_bench_step_per_chain(torch_dev, pool, bench_oracle, model, stream0):
    """one MYULA step of 64 chains at L = 256, B = 1.5 built as bench.py builds it (device Philox noise; stream0 = 64 is
    rank 1 of the weak-scaling run): every chain's gradient, prox support and signs, log pi terms and new state against
    numpy (R.soft, the Philox restatement, gradients by linearity), new predictions of the first and last chain of each
    128-column block against the oracle"""
    torch = torch_dev
    from oracle import pxmcmc_ref as R
    from pxmcmc_b200 import device as D
    from pxmcmc_b200.forward import RingPreds, SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1

    sig, real, fused = MODELS[model]
    d, ic, G, h = bench_oracle[model]
    a = chain_coefficients(NB, 64 + stream0, real=real)
    X = a @ bench_oracle["U"]
    op = SphericalWaveletTransformOperator(d, _ring_sigma() if sig == "ring" else sig, "synthesis", LB, BB, JB, nchains=NB)
    prm = PxMCMCParams(nsamples=1, nburn=0, ngap=1, delta=DELTA, lmda=LMDA, mu=1.0, verbosity=0, track=[])
    reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, LMDA, L=LB, B=BB, J_min=JB)
    outer = MYULA(op, reg, prm, noise="device", nchains=NB, seed=SEED, stream0=stream0, real_pairs=real)
    m = outer.engine
    m.forward.fuse_ring = m.forward.fuse_gram = fused
    Xd = D.to_dev_c(X)
    Xe = outer.pack(Xd) if real else Xd
    P = m._initial_preds(Xe)
    assert isinstance(P, RingPreds) == fused and (not fused or P.kind == "harm")
    if sig == "ring":
        assert isinstance(m.forward._gram_weights(), tuple)  # the weighted Gram table
    g = m.forward.gradg_from_ring(P) if fused else m.forward.calc_gradg(P)
    Ppix = m._pix(P)
    if real:
        g, Ppix = outer.unpack(g), outer.unpack(Ppix)
    g, prox = D.to_host(g), D.to_host(reg.proxf(Xd))
    lp, l2, pr = outer._logpi_dev(Xd, Ppix)
    Xn, Pn = m.iterate(Xe, P)
    Pn = m._pix(Pn)
    if real:
        Xn, Pn = outer.unpack(Xn), outer.unpack(Pn)
    Xn, Pn = D.to_host(Xn), D.to_host(Pn)
    torch.cuda.synchronize()
    # host restatement of the step
    prior = R.S2WaveletsL1("synthesis", None, None, LMDA, LB, BB, JB)
    o_prox = R.soft(X, prior.T)
    o_g = a @ G - h
    w = philox_ref.element_normals(2, NB, X.shape[1], SEED, 1, stream0)[0]
    o_Xn = R.myula_step(X, o_prox, o_g, DELTA, LMDA, w)
    PsiX = a @ bench_oracle["PsiU"]
    for c in range(NB):
        assert rel_l2(g[c], o_g[c]) < TOL, f"gradient chain {c}: {rel_l2(g[c], o_g[c]):.2e}"
        p, q = prox[c], o_prox[c]
        assert np.array_equal(p == 0, q == 0) and np.array_equal(np.sign(p.real), np.sign(q.real)) \
            and np.array_equal(np.sign(p.imag), np.sign(q.imag)), f"prox support / signs chain {c}"
        assert rel_l2(Xn[c], o_Xn[c]) < TOL, f"state chain {c}: {rel_l2(Xn[c], o_Xn[c]):.2e}"
        diff = d - PsiX[c]
        o_l2 = np.vdot(diff, ic * diff)
        o_pr = np.sum(np.abs(prior.map_weights * X[c]))
        assert np.isclose(l2[c], o_l2, rtol=1e-10, atol=0) and np.isclose(pr[c], o_pr, rtol=1e-12, atol=0), f"log pi terms chain {c}"
        assert np.isclose(lp[c], -o_pr - o_l2, rtol=1e-10, atol=0)
    assert 0 < np.count_nonzero(o_prox == 0) < o_prox.size  # the support comparison is not vacuous
    picks = (0, 31, 32, 63)
    for c, Po in zip(picks, pool.map(_w_oracle, [("inverse", o_Xn[c], LB, BB, JB) for c in picks])):
        assert rel_l2(Pn[c], Po) < TOL, f"predictions chain {c}: {rel_l2(Pn[c], Po):.2e}"


# ------------------------------------------------------------------ (c) Philox noise kernels against the restatement
def _assert_normals(got, ref, what):
    """a few ulp per normal (the device's log and sincospi are not correctly rounded; the restatement is)"""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, what
    tol = 8 * np.spacing(np.maximum(np.abs(ref), 1e-3))
    bad = np.abs(got - ref) > tol
    assert not bad.any(), f"{what}: {np.count_nonzero(bad)} normals off, first at {np.argwhere(bad)[0]}"


NOISE_CASES = [  # (n, chains, seed, step, stream0)
    (1, 3, 5, 1, 0),
    (7, 5, 2 ** 32 + 9, 2 ** 32 + 3, 2 ** 32 - 2),  # odd n, 64-bit step and seed, streams wrapping past 2^32
    (398342, 2, 1234, 7, 64),                       # one L = 256 wavelet state
    (3, 70000, 11, 5, 2 ** 32 - 40000),             # > 65 535 chains: the update launches in chain slices
]


@pytest.mark.parametrize("case", NOISE_CASES, ids=["n1", "odd-wide-counters", "L256", "70000-chains"])
@pytest.mark.parametrize("mode", [2, 3, 4])
def test_philox_update_noise_against_restatement(torch_dev, mode, case):
    """MYULA update with zero state and gradient and delta = 1/2 (sqrt(2 delta) = 1): X' = w exactly, through the plain,
    device-step (CUDA-graph) and per-chain-parameter (PxMALA) forms of the kernel"""
    torch = torch_dev
    from pxmcmc_b200 import device as D

    n, nch, seed, step, stream0 = case
    w_re, w_im = philox_ref.element_normals(mode, nch, n, seed, step, stream0)
    zero = torch.zeros((nch, n), dtype=torch.complex128, device="cuda")
    outs = {"step": D.myula_update_dev(zero, None, zero, None, 0.0, 0.5, 1.0, noise_mode=mode, seed=seed, step=step,
                                       stream0=stream0)}
    dstep = torch.tensor([step], dtype=torch.int64, device="cuda")
    outs["dstep"] = D.myula_update_dev(zero, None, zero, None, 0.0, 0.5, 1.0, noise_mode=mode, seed=seed, stream0=stream0,
                                       dstep=dstep)
    assert int(dstep.item()) == step + 1
    if mode != 4:  # (PxMALA's per-chain step sizes: its chains are complex, never packed real pairs)
        S = torch.zeros((nch, 16), dtype=torch.float64, device="cuda")
        S[:, 0], S[:, 1], S[:, 2], S[:, 3] = 0.5, 0.5, 0.5, 1.0
        S[:, 14] = float(step)  # step 0 passed: the kernel reads it from the state block, as in a captured PxMALA loop
        outs["dpar"] = D.myula_update_dpar_dev(zero, None, zero, None, 0.0, S, mode, seed, 0, stream0)
    for form, x in outs.items():
        x = D.to_host(x)
        _assert_normals(x.real, w_re, f"mode {mode}, {form}, real part")
        if mode == 2:
            assert np.all(x.imag == 0), f"mode 2, {form}: real noise only"
        else:
            _assert_normals(x.imag, w_im, f"mode {mode}, {form}, imaginary part")


@pytest.mark.parametrize("case", NOISE_CASES, ids=["n1", "odd-wide-counters", "L256", "70000-chains"])
def test_philox_normal_kernel_against_restatement(torch_dev, case):
    """SKROCK's normals (`k_philox_normal`), with the step given and read from the device"""
    torch = torch_dev
    from pxmcmc_b200 import device as D

    n, nch, seed, step, stream0 = case
    ref = philox_ref.element_normals(2, nch, n, seed, step, stream0)[0]
    _assert_normals(D.to_host(D.philox_normal_dev(nch, n, seed, step, stream0)), ref, "k_philox_normal")
    dstep = torch.tensor([step], dtype=torch.int64, device="cuda")
    _assert_normals(D.to_host(D.philox_normal_dev(nch, n, seed, 0, stream0, dstep=dstep)), ref, "k_philox_normal, device step")


# ------------------------------------------------------------------ (d) CSR SpMV against scipy
@pytest.mark.parametrize("nch", [1, 2, 3, 4, 5, 9, 64])
def test_csr_spmv_against_scipy(torch_dev, nch):
    """real CSR matrix times complex chains (warp per row; groups of four chains per warp with full and partial groups):
    rows without entries, rows of more than 32 entries (several passes of the warp), per chain"""
    torch = torch_dev
    from pxmcmc_b200 import device as D

    rng = np.random.default_rng(nch)
    nrows, ncols = 70, 500
    counts = rng.integers(0, 12, nrows)
    counts[[0, 5, 6, 69]] = 0
    counts[[1, 30]] = [33, 200]
    counts[2] = 64
    rows = np.repeat(np.arange(nrows), counts)
    cols = np.concatenate([rng.choice(ncols, k, replace=False) for k in counts])
    A = sparse.csr_matrix((rng.standard_normal(rows.size), (rows, cols)), shape=(nrows, ncols))
    A.sort_indices()
    assert np.diff(A.indptr).max() == 200 and np.count_nonzero(np.diff(A.indptr) == 0) >= 4
    x = _crandn(rng, nch, ncols) * np.logspace(0, -6, nch)[:, None]
    dev = lambda v, t: torch.from_numpy(np.ascontiguousarray(v, dtype=t)).cuda()  # noqa: E731
    y = D.to_host(D.csr_spmv_dev(dev(A.indptr, np.int32), dev(A.indices, np.int32), dev(A.data, np.float64),
                                 D.to_dev_c(x), nrows, ncols))
    exp = (A @ x.T).T
    for c in range(nch):
        assert rel_l2(y[c], exp[c]) < 1e-14, f"chain {c}"
        assert np.all(y[c][np.diff(A.indptr) == 0] == 0)
