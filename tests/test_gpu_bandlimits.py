"""GPU parity at the bandlimits where the kernels change (`pytest -m gpu`).

The ring of bandlimit l has n = 2l - 1 points and Bluestein length M = the smallest power of two >= 2n - 1.  M picks the
ring-FFT kernel: M <= 256 (l <= 64) the two-pass class-0 kernel, M = 512 / 1024 (l <= 256) the persistent staged kernel
on wide grids, M = 2048 / 4096 (l <= 1024) the multi-pass kernel, which a wide grid launches beside the other two on the
same stage (`min_logM = 11`).  A grid below 700 CTAs runs every class on the multi-pass kernel.  Every boundary pair
64/65 ... 512/513 and L = 1024 is checked here against the CPU oracle, chain by chain, at one chain and at 64/65.

The device builds its Legendre tables Lambda^{m,s}_l(theta_t) = (-1)^s sqrt((2l+1)/4pi) d^l_{m,-s}(theta_t) at plan
creation with a recurrence in l (pxm_wigner.cuh).  They are checked through the public inverse SHT of unit
coefficients against Wigner's explicit sum in arbitrary precision (oracle/wigner_mp.py), at L = 1024 and 513, at the
rings next to both poles and to the equator, and on HEALPix rings.

Oracle calls run in CPU worker processes, all submitted when the module starts so that the slow L = 1024 ones overlap
the GPU work of the others.
"""
import os
from concurrent.futures import ProcessPoolExecutor
import multiprocessing as mp

import numpy as np
import pytest

from conftest import rel_l2
from test_gpu_batch_widths import _poison_allocator, _w_oracle, _with_debug, chain_coefficients

pytestmark = pytest.mark.gpu

TOL = 1e-10
K = 3
J_MIN = 2
BOUNDARY_L = [64, 65, 128, 129, 256, 257, 512, 513, 1024]
WIDE = (64, 65)
SMALL_GRID_CTAS = 700  # pxm_fft_launch: below this many CTAs every class runs on the multi-pass kernel

WAV_CASES = [(L, 2.0, nb) for L in BOUNDARY_L for nb in ((1,) + WIDE if L <= 513 else (1,))]
WAV_CASES += [(257, 1.5, nb) for nb in (1,) + WIDE]
SHT_CASES = [(L, s, nb) for L in BOUNDARY_L if L <= 513 for s in (0, 2) for nb in (1,) + WIDE] + [(1024, 0, 1)]
WAVELET_OPS = {"synthesis": ("coef", "inverse"), "synthesis_adjoint": ("pix", "inverse_adjoint"),
               "analysis": ("pix", "forward"), "analysis_adjoint": ("coef", "forward_adjoint")}
SHT_FNS = {"inverse": "flm", "forward": "pix", "inverse_adjoint": "pix", "forward_adjoint": "flm"}


# ------------------------------------------------------------------ ring-FFT dispatch restated (pxm_fft.cu)
def bluestein_logM(ell):
    """pxm_fft_choose_M: the smallest power of two >= 2n - 1 (at least 16) for the ring of n = 2 ell - 1 points"""
    n, lg = 2 * ell - 1, 4
    while (1 << lg) < 2 * n - 1:
        lg += 1
    return lg


def rings_per_cta_log(logM):
    """pxm_fft_rings_per_cta_log: 4096 points per CTA, at most 16 rings"""
    lg = 0
    while ((1 << logM) << (lg + 1)) <= 4096 and lg < 4:
        lg += 1
    return lg


def class_bit(logM):
    """pxm_fft_class_bit: 1 two-pass (M <= 256), 2 persistent / two-pass (M = 512, 1024), 4 multi-pass (M > 1024)"""
    return 1 if logM <= 8 else (2 if logM <= 10 else 4)


def fft_stage(bandlimits):
    """(CTAs of one chain, class mask) of a ring-FFT stage over the ring grids of these bandlimits"""
    ctas, mask = 0, 0
    for ell in bandlimits:
        lg = bluestein_logM(ell)
        ctas += -(-ell // (1 << rings_per_cta_log(lg)))
        mask |= class_bit(lg)
    return ctas, mask


def test_dispatch_restatement_at_the_class_boundaries():
    """the restated Bluestein lengths change class where the module docstring says (no device needed)"""
    assert [1 << bluestein_logM(ell) for ell in BOUNDARY_L] == [256, 512, 512, 1024, 1024, 2048, 2048, 4096, 4096]
    assert [class_bit(bluestein_logM(ell)) for ell in (64, 65, 256, 257, 1024)] == [1, 2, 2, 4, 4]
    assert fft_stage([257]) == (129, 4) and fft_stage([64]) == (4, 1)


# ------------------------------------------------------------------ oracle workers (CPU processes)
def _w_wigner_column(args):
    """Lambda^{m,s}_l at a list of MW rings (p_t = 2t + 1, q = 2L - 1) or HEALPix rings (sin^2(theta/2)), mpf"""
    l, m, s, thetas = args
    from oracle import wigner_mp as W

    return [W.wigner_d(l, m, -s, *th) if isinstance(th, tuple) else W.wigner_d_sin2(l, m, -s, th) for th in thetas]


@pytest.fixture(scope="module")
def pool():
    n = max(1, min(8, (os.cpu_count() or 2) - 1))
    ex = ProcessPoolExecutor(n, mp_context=mp.get_context("spawn"))
    yield ex
    ex.shutdown(wait=True, cancel_futures=True)  # (after a failure: no waiting for results nobody reads)


@pytest.fixture(scope="module")
def torch_dev():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def _nbasis(L):
    return 1 if L > 513 else K  # L = 1024 runs one chain: one basis input per operator


def _basis(L, kind, n, tag):
    """basis inputs [K, n] of one input kind, seeded by the case (flm of spin 2: l < 2 zero)"""
    rng = np.random.default_rng([L, int(10 * tag), ["coef", "pix", "flm"].index(kind)])
    u = _crandn(rng, _nbasis(L), n)
    if kind == "flm" and tag == 2:
        u[:, :4] = 0
    return u


# ------------------------------------------------------------------ Legendre-table cases
TABLE_CASES = [(1024, 0), (1024, 2), (1024, -2), (513, 0), (513, 2)]
# per value, times sqrt((2l+1)/4pi); the worst seen on a B200 was 8.3e-13 (L = 1024, spin +-2), so the bar is the
# host-recurrence test's 1e-11 rather than 1e-12
TABLE_TOL = 1e-11
HPX_NSIDE, HPX_L = 256, 256


def table_pairs(L, s):
    """(l, m) of the unit coefficients: the first and last degrees and the middle one, m at 0, +-1, +-l/2, +-(l-1),
    +-l (m = l = L - 1 is the deepest underflowing seed; m = 0, +-1 are the |m| < |s| cases of spin 2)"""
    a = abs(s)
    pairs = set()
    for l in (a, a + 1, L // 2, L - 2, L - 1):
        for m in (0, 1, l // 2, l - 1, l):
            for sg in (1, -1):
                if abs(m) <= l:
                    pairs.add((l, sg * m))
    return sorted(pairs)


# a ring where the seed of m = l/2 (l = L - 1 or L - 2) is below e^-600, carried with a binary exponent, and the row
# grows back past 1e-200 by l = L - 1: the 2^300 rescale runs with a nonzero exponent
RESCALE_RING = {1024: 96, 513: 12}


def table_rings(L):
    """t = 0 ... 7 and L - 8 ... L - 1 (t = L - 1 is theta = pi), the rings on either side of sin^2(theta/2) = 0.5, the
    rescale ring and 16 seeded random rings"""
    lo = (2 * L - 3) // 4  # last ring with theta < pi/2: 2 (2t + 1) < 2L - 1
    assert 2 * (2 * lo + 1) < 2 * L - 1 < 2 * (2 * lo + 3)
    rings = set(range(8)) | set(range(L - 8, L)) | {lo, lo + 1, RESCALE_RING[L]}
    rest = np.setdiff1d(np.arange(L), sorted(rings))
    rings |= set(np.random.default_rng(L).choice(rest, 16, replace=False).tolist())
    return sorted(rings)


def hpx_pairs(L):
    return table_pairs(L, 0)


def hpx_rings(nside):
    return [1, 2, nside - 1, nside, 2 * nside, 3 * nside, 4 * nside - 1]


# ------------------------------------------------------------------ every oracle job, submitted at once
@pytest.fixture(scope="module")
def jobs(pool, request):
    """futures of the oracle results the selected tests of this module need; the slowest first"""
    from oracle import pxmcmc_ref as R
    from oracle import wigner_mp as W

    sel = {}
    for it in request.session.items:
        if it.module.__name__ == __name__:
            params = tuple(it.callspec.params.values()) if hasattr(it, "callspec") else ()
            sel.setdefault(it.originalname, set()).add(params)
    wav = sel.get("test_wavelet_operators_at_class_boundaries", set())
    sht = sel.get("test_sht_at_class_boundaries", set())
    fut = {}
    # transforms at L = 1024 (minutes each), then the Legendre columns, then the boundary transforms in test order
    order = sorted({L for L, _, _ in wav} | {L for L, _, _ in sht}, key=lambda L: (L != 1024, L))
    for L in order[:1]:
        _submit_transforms(pool, fut, L, R, wav, sht)
    for L, s in sorted(sel.get("test_legendre_tables_against_wigner_explicit_sum", set())):
        rings = [(2 * t + 1, 2 * L - 1) for t in table_rings(L)]
        for l, m in table_pairs(L, s):
            fut[("table", L, s, l, m)] = pool.submit(_w_wigner_column, (l, m, s, rings))
    if "test_healpix_rows_against_wigner_explicit_sum" in sel:
        hr = [W.healpix_sin2_half(HPX_NSIDE, i) for i in hpx_rings(HPX_NSIDE)]
        for l, m in hpx_pairs(HPX_L):
            fut[("hpx", l, m)] = pool.submit(_w_wigner_column, (l, m, 0, hr))
    for L in order[1:]:
        _submit_transforms(pool, fut, L, R, wav, sht)
    return fut


def _submit_transforms(pool, fut, L, R, wav, sht):
    for B in sorted({B for LL, B, _ in wav if LL == L}):
        ncoefs = R.WaveletTransform(L, B, J_MIN).ncoefs
        U = {"coef": _basis(L, "coef", ncoefs, B), "pix": _basis(L, "pix", L * (2 * L - 1), B)}
        for name, (kind, op) in WAVELET_OPS.items():
            fut[("wav", L, B, name)] = (U[kind], [pool.submit(_w_oracle, (op, u, L, B, J_MIN)) for u in U[kind]])
    for s in sorted({s for LL, s, _ in sht if LL == L}):
        U = {"flm": _basis(L, "flm", L * L, s), "pix": _basis(L, "pix", L * (2 * L - 1), s)}
        for fn, kind in SHT_FNS.items():
            fut[("sht", L, s, fn)] = (U[kind], [pool.submit(_w_oracle, (f"sht{s}_{fn}", u, L, 0, 0)) for u in U[kind]])


def _result(fut, key):
    """(basis inputs [K, n], oracle outputs [K, n_out])"""
    U, fs = fut[key]
    return U, np.stack([np.asarray(f.result()).ravel() for f in fs])


# ------------------------------------------------------------------ (a) Legendre tables against Wigner's explicit sum
def _check_rows(got, refs, l, m, s, sin_theta, phases, what):
    """got [rings, ncol] complex, refs: mpf per ring, sin_theta: per ring, phases [rings, ncol]: e^{i m phi} of each
    column; returns the worst |error| / sqrt((2l+1)/4pi)"""
    norm = np.sqrt((2 * l + 1) / (4 * np.pi))
    tiny = np.finfo(np.float64).tiny
    worst = 0.0
    for r, ref in enumerate(refs):
        row = got[r]
        if 0 < abs(ref) < tiny:  # the true value underflows: zero or subnormal, never a normal number
            assert np.all(np.abs(row.real) < tiny) and np.all(np.abs(row.imag) < tiny), \
                f"{what}, ring {r}: true |value| {float(abs(ref)):.1e} below DBL_MIN, got {np.abs(row).max():.3e}"
            continue
        v = float(ref)
        e0 = abs(row[0] - v * phases[r][0])  # the first column: the table entry itself
        e = np.abs(row - v * phases[r]).max()  # the whole ring: the ring FFT of a single m
        worst = max(worst, e0 / norm, e / norm)
        # absolute bar, and relative for tiny values in the polar part of a row before its turning point (monotone,
        # where a wrong power of two in the exponent tracking would hide under the absolute bar; not the zeros of the
        # oscillating part, such as l + m odd at theta = pi/2)
        bar = TABLE_TOL * norm
        if 1e-280 < abs(v) < 1e-30 and (l + 0.5) * sin_theta[r] < max(abs(m), abs(s)):
            bar = min(bar, 1e-10 * abs(v))
        assert e0 <= bar and e <= bar, \
            f"{what}, ring {r}: ref {v:.17e}, first column {row[0]:.17e}, ring error {e:.2e} (bar {bar:.2e})"
    return worst


@pytest.mark.parametrize("L,spin", TABLE_CASES, ids=[f"L{L}-s{s}" for L, s in TABLE_CASES])
def test_legendre_tables_against_wigner_explicit_sum(torch_dev, jobs, L, spin):
    """inverse SHT of unit coefficients, one (l, m) per chain: ring t of chain (l, m) is Lambda^{m,s}_l(theta_t)
    e^{i m phi_p}.  Each value within 1e-11 sqrt((2l+1)/4pi) of the arbitrary-precision value (and within 1e-10
    relative between 1e-280 and 1e-30 before a row's turning point), nonzero true values below DBL_MIN zero or
    subnormal.  Seeds below DBL_MIN
    (m = l = L - 1 at the polar rings), the 2^300 rescale, both half-angle forms of the recurrence coefficient,
    theta = pi and the device sincospi / lgamma are all on this path.  Worst seen on a B200 (1000 W): 8.3e-13 of
    sqrt((2l+1)/4pi) at L = 1024, spin +-2; 7.7e-13 at L = 513, spin 0."""
    torch = torch_dev
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D

    pairs, rings = table_pairs(L, spin), table_rings(L)
    n = 2 * L - 1
    plan = D.ShtPlan(L, spin, len(pairs))  # not cached: the tables go with the plan
    try:
        flm = torch.zeros((len(pairs), L * L), dtype=torch.complex128, device="cuda")
        for c, (l, m) in enumerate(pairs):
            flm[c, l * l + l + m] = 1
        f = plan.inverse(flm).reshape(len(pairs), L, n)
        got = D.to_host(f[:, torch.tensor(rings, device="cuda")])
        del f, flm
    finally:
        _lib.check(_lib.lib.pxm_sht_plan_destroy(plan.h))
        plan.h = None
    p = np.arange(n)
    sin_t = np.sin(np.pi * (2 * np.array(rings) + 1) / n)
    worst = 0.0
    for c, (l, m) in enumerate(pairs):
        d = jobs[("table", L, spin, l, m)].result()
        refs = [(-1) ** (abs(spin) & 1) * mp_norm(l) * x for x in d]
        phases = np.exp(2j * np.pi * ((m * p) % n) / n)[None, :].repeat(len(rings), 0)
        worst = max(worst, _check_rows(got[c], refs, l, m, spin, sin_t, phases, f"L={L} s={spin} l={l} m={m}"))
    print(f"\nLegendre tables L={L} spin={spin}: worst |error| / sqrt((2l+1)/4pi) = {worst:.2e}")


def mp_norm(l):
    import mpmath

    with mpmath.workdps(50):
        return mpmath.sqrt(mpmath.mpf(2 * l + 1) / (4 * mpmath.pi))


def test_healpix_rows_against_wigner_explicit_sum(torch_dev, jobs):
    """the same check through the HEALPix synthesis (nside = 256, L = 256), whose tables take their half angles from
    the exact z of the ring (1 - z = 1 / (3 nside^2) at the first ring) rather than from the MW formula"""
    from oracle import healpix_ref
    from oracle import wigner_mp as W
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D
    from pxmcmc_b200 import utils

    nside, L = HPX_NSIDE, HPX_L
    table = healpix_ref.ring_table(nside)
    rings = hpx_rings(nside)
    plan = utils._HealpixPlan(nside, L)  # not cached
    worst = 0.0
    try:
        for l, m in hpx_pairs(L):
            flm = np.zeros(L * L, complex)
            flm[l * l + l + m] = 1
            mp_map = D.to_host(plan.synth(D.to_dev_c(flm)))
            refs = [mp_norm(l) * x for x in jobs[("hpx", l, m)].result()]
            rows, phases = [], []
            for i in rings:
                npr, start, shift, _ = table[i - 1]
                rows.append(mp_map[start:start + npr])
                phases.append(np.exp(1j * m * (np.arange(npr) + 0.5 * shift) * 2 * np.pi / npr))
            for r in range(len(rings)):  # ragged rings: one at a time
                s2 = float(W.healpix_sin2_half(nside, rings[r]))
                worst = max(worst, _check_rows(rows[r][None], refs[r:r + 1], l, m, 0, [2 * np.sqrt(s2 * (1 - s2))],
                                               phases[r][None], f"HEALPix ring {rings[r]} l={l} m={m}"))
    finally:
        _lib.check(_lib.lib.pxm_hpx_plan_destroy(plan.h))
        plan.h = None
    print(f"\nHEALPix rows nside={nside} L={L}: worst |error| / sqrt((2l+1)/4pi) = {worst:.2e}")


# ------------------------------------------------------------------ (b) transforms at the class boundaries
def _per_chain(got, exp, what, a):
    worst = 0.0
    assert got.shape == exp.shape, what
    for c in range(got.shape[0]):
        err = rel_l2(got[c], exp[c])
        worst = max(worst, err)
        assert err < TOL, f"{what}, chain {c} (scale {np.abs(a[c]).max():.0e}): rel-L2 {err:.2e}"
    return worst


def _nan_call(torch, fn, x, n_out):
    """fn(x) writing into a caller buffer of NaN (the kernels must write every element)"""
    from pxmcmc_b200 import device as D

    buf = torch.full((x.shape[0], n_out), complex("nan+nanj"), dtype=torch.complex128, device="cuda")
    with D.output_into(buf):
        out = fn(x)
    assert out.data_ptr() == buf.data_ptr()
    return out


def _inputs(a, U):
    from pxmcmc_b200 import device as D

    return D.to_dev_c(a @ U)


@pytest.mark.parametrize("L,B,nb", WAV_CASES, ids=[f"L{L}-B{B}-nb{nb}" for L, B, nb in WAV_CASES])
def test_wavelet_operators_at_class_boundaries(torch_dev, jobs, L, B, nb):
    """all four wavelet operators (B = 2, J_min = 2: the scales of one plan span several FFT classes) at one chain and
    at 64 / 65 chains against the oracle, rel-L2 < 1e-10 per chain.  From the host: which ring-FFT path the stage took
    (a wide grid above L = 256 mixes the multi-pass class-4 groups with the persistent and class-0 kernels); at 257 and
    513 the default equals the forced persistent mode bit for bit and the all-multi-pass mode to 1e-13.  Worst rel-L2
    seen on a B200: 9.3e-13 up to L = 513, 1.9e-12 at L = 1024."""
    torch = torch_dev
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D

    plan = D.WaveletPlan(L, B, J_MIN, nb)  # not cached
    try:
        ctas, mask = fft_stage(plan.bandlimits)
        if nb in WIDE:
            assert ctas * nb >= SMALL_GRID_CTAS, "the wide case no longer reaches the split ring-FFT dispatch"
            if L > 256:
                assert mask & 4 and mask & 3, f"scales {plan.bandlimits}: no mixed class-4 stage (mask {mask})"
        elif L <= 512:
            assert ctas * nb < SMALL_GRID_CTAS, "one chain no longer runs the multi-pass kernel"
        a = chain_coefficients(nb, 7 * L + nb)[:, :_nbasis(L)]
        res = {name: _result(jobs, ("wav", L, B, name)) for name in WAVELET_OPS}
        X = {name: _inputs(a, U) for name, (U, _) in res.items()}

        def run():
            _poison_allocator(torch, 16 * nb * max(plan.ncoefs, plan.npix))
            n_out = {"synthesis": plan.npix, "synthesis_adjoint": plan.ncoefs, "analysis": plan.ncoefs,
                     "analysis_adjoint": plan.npix}
            out = {name: D.to_host(_nan_call(torch, getattr(plan, name), X[name], n_out[name])) for name in WAVELET_OPS}
            torch.cuda.synchronize()
            return out

        got = run()
        worst = max(_per_chain(got[name], a @ res[name][1], f"{name} L={L} B={B} nb={nb}", a) for name in WAVELET_OPS)
        print(f"\nwavelet L={L} B={B} nb={nb} scales={plan.bandlimits} stage ctas/chain={ctas} mask={mask}: "
              f"worst rel-L2 {worst:.2e}")
        if nb == 64 and L in (257, 513):
            forced = _with_debug(run, fft=3)
            multi = _with_debug(run, fft=1)
            for name in WAVELET_OPS:
                assert np.array_equal(got[name], forced[name]), f"{name}: default ring FFT is not the split dispatch"
                for c in range(nb):
                    assert rel_l2(got[name][c], multi[name][c]) < 1e-13, f"{name} chain {c}: split vs multi-pass"
    finally:
        _lib.check(_lib.lib.pxm_wav_plan_destroy(plan.h))
        plan.h = None


@pytest.mark.parametrize("L,spin,nb", SHT_CASES, ids=[f"L{L}-s{s}-nb{nb}" for L, s, nb in SHT_CASES])
def test_sht_at_class_boundaries(torch_dev, jobs, L, spin, nb):
    """the four SHTs of one bandlimit (one ring grid) at one chain and at 64 / 65 chains against the oracle,
    rel-L2 < 1e-10 per chain (worst seen on a B200: 3.4e-13 up to L = 513, 7.3e-13 at L = 1024)"""
    torch = torch_dev
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D

    plan = D.ShtPlan(L, spin, nb)  # not cached
    try:
        a = chain_coefficients(nb, 11 * L + nb + spin)[:, :_nbasis(L)]
        _poison_allocator(torch, 16 * nb * plan.npix)
        worst = 0.0
        for fn, kind in SHT_FNS.items():
            U, T = _result(jobs, ("sht", L, spin, fn))
            n_out = plan.nlm if kind == "pix" else plan.npix
            got = D.to_host(_nan_call(torch, getattr(plan, fn), _inputs(a, U), n_out))
            worst = max(worst, _per_chain(got, a @ T, f"SHT {fn} L={L} spin={spin} nb={nb}", a))
        print(f"\nSHT L={L} spin={spin} nb={nb}: worst rel-L2 {worst:.2e}")
    finally:
        _lib.check(_lib.lib.pxm_sht_plan_destroy(plan.h))
        plan.h = None


# ------------------------------------------------------------------ (c) above the range
def test_bandlimit_above_1024_is_refused_cleanly(torch_dev):
    """L = 1025 would need Bluestein length 8192: plan creation refuses it with the library's error before it allocates
    anything, and a following plan still works"""
    from pxmcmc_b200 import _lib
    from pxmcmc_b200 import device as D

    for make in (lambda: D.ShtPlan(1025, 0, 1), lambda: D.WaveletPlan(1025, 2.0, J_MIN, 1)):
        with pytest.raises(_lib.PxmError, match=r"L must be in \[\d, 1024\]"):
            make()
    plan = D.ShtPlan(64, 0, 1)
    try:
        flm = np.zeros(64 * 64, complex)
        flm[0] = 1
        f = D.to_host(plan.inverse(D.to_dev_c(flm)))
        assert np.allclose(f, 1 / np.sqrt(4 * np.pi), rtol=0, atol=1e-15)
    finally:
        _lib.check(_lib.lib.pxm_sht_plan_destroy(plan.h))
        plan.h = None
