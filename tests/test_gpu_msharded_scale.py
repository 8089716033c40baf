"""GPU parity of the m-sharded weak-lensing chain at the size `bench.py` runs it (config 4: L = 512, B = 2, J_min = 2).

All ranks run in one process on one GPU through `msharded.SimulatedRanks` (one stream per rank, the same peer
pointers, push / pull contractions and flag barrier as one process per GPU).  The expected values come from the
unsharded plans and samplers, which test_gpu_configs.py pins to the CPU oracle at L = 512.

1. The transforms at L = 257, 512 and 513 on 2 and 3 ranks, on 8 ranks at L = 257, and with 64 chains per plan at
   L = 257.  A rank's ring FFT covers only its own 64-ring blocks, so its grid can fall on the other side of the
   700-CTA dispatch threshold than the unsharded grid: the sharded result then comes from other ring-FFT kernels than
   the one it must match.  The host restatement of that dispatch below names the cases where this happens.
2. The sampler's own iteration (`MYULA.iterate`, Philox noise drawn on the device, stream0 = rank) enqueued five times
   back to back with no host synchronisation, so that iteration k + 1 of one rank overlaps iteration k of the others
   and only the peer barriers keep the ring buffers apart.
   Expected: the unsharded sampler stepped with the same normals, restated on the host (oracle/philox_ref.py) rank
   by rank.  This first test of `MYULA.iterate` under `SimulatedRanks` found that the sharded prior uploaded its
   thresholds on first use, a blocking copy that waited on a barrier whose peers were not enqueued yet.
3. The same iteration captured as one CUDA graph per rank and replayed: the barrier epochs must come from device
   memory.
4. One process per GPU (torchrun, CUDA IPC), `scripts/msharded_check.py --iterate`, skipped below two GPUs.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, rel_l2
from oracle import philox_ref
from test_gpu_bandlimits import SMALL_GRID_CTAS, bluestein_logM, class_bit, fft_stage, rings_per_cta_log
from test_gpu_batch_widths import chain_coefficients

pytestmark = pytest.mark.gpu

B, J_MIN = 2.0, 2
TOL = 1e-13  # sharded against unsharded: the same kernels and summation order, up to the ring-FFT kernel choice
# 8 ranks at L = 512 and 513 agree as well (worst 6.0e-16 and 1.0e-15 on a B200) but take 55 s each: 8 ranks are
# covered at L = 257, where the ring grids have fewer 64-ring blocks than ranks
TRANSFORM_CASES = [(L, world) for L in (257, 512, 513) for world in (2, 3)] + [(257, 8)]
WIDE_CASES = [(257, 2), (257, 8)]
NB_WIDE = 64
WAVELET_OPS = {"synthesis": ("coef", "pix"), "synthesis_adjoint": ("pix", "coef"), "analysis": ("pix", "coef"),
               "analysis_adjoint": ("coef", "pix"), "synthesis_harmonic": ("coef", "flm0"),
               "synthesis_adjoint_harmonic": ("flm0", "coef")}
SHT_OPS = {"inverse": ("flm", "pix"), "forward": ("pix", "flm"), "inverse_adjoint": ("pix", "flm"),
           "forward_adjoint": ("flm", "pix")}


def bandlimits(L):
    """the wavelet plan's ring grids: scaling function, then wavelet scales J_min ... J (pxm_wav_plan_bandlimits)"""
    J = int(np.ceil(np.log(L) / np.log(B)))
    return [min(int(np.ceil(B ** J_MIN)), L)] + [min(int(np.ceil(B ** (j + 1))), L) for j in range(J_MIN, J + 1)]


# ------------------------------------------------------------------ ring-FFT dispatch of one rank, restated on the host
def rank_stage(grids, rank, world):
    """(CTAs of one chain, class mask) of the ring-FFT stage of `rank` over these (bandlimit, rotation) grids: only the
    rows `ring_range` gives the rank (add_fft_group in pxm_plan.cu); world = 1 is `fft_stage` of test_gpu_bandlimits.py"""
    from pxmcmc_b200 import msharded as ms

    ctas, mask = 0, 0
    for ell, rot in grids:
        t0, t1 = ms.ring_range(ell, rot, rank, world)
        if t1 > t0:
            lg = bluestein_logM(ell)
            ctas += -(-(t1 - t0) // (1 << rings_per_cta_log(lg)))
            mask |= class_bit(lg)
    return ctas, mask


def dispatch(ctas, mask, nb):
    """which ring-FFT kernels a stage of `nb` chains runs (pxm_fft_launch)"""
    if ctas == 0:
        return "none"
    return "multi-pass" if ctas * nb < SMALL_GRID_CTAS and mask & 6 else "split"


def stages(L):
    """the ring-FFT stages of the three plans of an iteration: wavelet scales, wavelet / SHT full grid"""
    bl = bandlimits(L)
    return {"scales": [(ell, i + 1) for i, ell in enumerate(bl)], "full": [(L, 0)]}


def dispatch_mismatches(L, world, nb):
    """[(stage, rank, unsharded kernels, rank's kernels)] where a rank runs other ring-FFT kernels than the plan it
    must match (ranks that own no ring of the grid launch nothing and are left out)"""
    out = []
    for name, grids in stages(L).items():
        whole = dispatch(*fft_stage([ell for ell, _ in grids]), nb)
        for r in range(world):
            mine = dispatch(*rank_stage(grids, r, world), nb)
            if mine not in ("none", whole):
                out.append((name, r, whole, mine))
    return out


def test_dispatch_restatement_finds_sharded_unsharded_splits():
    """The chosen cases include stages where the unsharded plan is at or above 700 CTAs and a rank below.  At one chain
    this already happens at L = 513: its scale grids (512, 513, 513) give the unsharded stage 1 371 CTAs, every rank of
    3 (and of 8) and rank 1 of 2 stay below 700.  At 64 chains on 8 ranks (L = 257) the rank holding the last single
    ring of the full grid launches 64 CTAs, and rank 6 of the scales holds only M = 512 rings (class bit 2, 8 CTAs a
    chain)."""
    from pxmcmc_b200 import msharded  # noqa: F401  (ring_range: host-only library call)

    assert fft_stage([ell for ell, _ in stages(513)["scales"]]) == (1371, 7)
    found = {(L, w, 1): dispatch_mismatches(L, w, 1) for L, w in TRANSFORM_CASES}
    found.update({(L, w, NB_WIDE): dispatch_mismatches(L, w, NB_WIDE) for L, w in WIDE_CASES})
    for key, mm in found.items():
        if mm:
            print(f"\nL={key[0]} world={key[1]} nb={key[2]}: " + "; ".join(f"{s} rank {r}: {a} unsharded, {b} sharded"
                                                                            for s, r, a, b in mm))
    assert ("scales", 1, "split", "multi-pass") in found[(513, 2, 1)]
    assert found[(513, 3, 1)] == [("scales", r, "split", "multi-pass") for r in range(3)]
    assert ("full", 4, "split", "multi-pass") in found[(257, 8, NB_WIDE)]
    assert ("scales", 6, "split", "multi-pass") in found[(257, 8, NB_WIDE)]
    # below L = 513 one chain runs the multi-pass kernel on both sides
    assert not any(found[(L, w, 1)] for L, w in TRANSFORM_CASES if L < 513)


# ------------------------------------------------------------------ fixtures and helpers
@pytest.fixture(scope="module")
def ms():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pxmcmc_b200 import device as D
    from pxmcmc_b200 import msharded

    cached = (set(D.WaveletPlan._cache), set(D.ShtPlan._cache))
    yield msharded
    # plans hold their Legendre tables until destroyed: release the cached ones this module created
    from pxmcmc_b200 import _lib

    torch.cuda.synchronize()
    for cls, before, kind in ((D.WaveletPlan, cached[0], "wav"), (D.ShtPlan, cached[1], "sht")):
        for key in set(cls._cache) - before:
            _lib.check(getattr(_lib.lib, f"pxm_{kind}_plan_destroy")(cls._cache.pop(key).h))


def _destroy(*plans):
    from pxmcmc_b200 import _lib

    for p in plans:
        if p is not None and p.h is not None:
            kind = "wav" if hasattr(p, "bandlimits") else "sht"
            _lib.check(getattr(_lib.lib, f"pxm_{kind}_plan_destroy")(p.h))
            p.h = None


def _destroy_sim(sim):
    import torch

    torch.cuda.synchronize()
    for plans in sim.plan_sets:
        _destroy(*plans)


def _crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def _host(t):
    return t.detach().cpu().numpy()


def _basis(L, ncoefs, nrows, seed):
    """inputs of every kind, [nrows, n]; spin-2 f_lm have l < 2 zero"""
    rng = np.random.default_rng(seed)
    U = {"coef": _crandn(rng, nrows, ncoefs), "pix": _crandn(rng, nrows, L * (2 * L - 1)),
         "flm0": _crandn(rng, nrows, L * L), "flm2": _crandn(rng, nrows, L * L)}
    U["flm2"][:, :4] = 0
    return U, rng.standard_normal(L)


def _unsharded(L, nb, U, gl):
    """every operation of the unsharded plans of nb chains on the inputs U: {op: [nb, n_out]}"""
    from pxmcmc_b200 import device as D

    wp, s0, s2 = D.WaveletPlan(L, B, J_MIN, nb), D.ShtPlan(L, 0, nb), D.ShtPlan(L, 2, nb)
    try:
        out = {}
        for name, (kin, _) in WAVELET_OPS.items():
            out[name] = _host(getattr(wp, name)(D.to_dev_c(U[kin])))
        for spin, plan in ((0, s0), (2, s2)):
            for fn, (kin, _) in SHT_OPS.items():
                for g in (None, gl):
                    x = U[f"flm{spin}"] if kin == "flm" else U["pix"]
                    out[(spin, fn, g is not None)] = _host(getattr(plan, fn)(D.to_dev_c(x), gl=None if g is None else D.to_dev_f(g)))
        return out, wp.ncoefs, wp.bandlimits
    finally:
        _destroy(wp, s0, s2)


def _run_sharded(ms, sim, plans, method, kin, kout, full_in, L, gl=None):
    """plans[r].<method> on every rank, inputs cut from full_in [nb, n]; returns the full output [nb, n_out].  Harmonic
    inputs hold NaN in the orders a rank does not own; harmonic outputs must hold exact zeros there."""
    from pxmcmc_b200 import device as D

    world = sim.world
    masks = [ms.flm_owner_mask(L, r, world) for r in range(world)]
    ins = []
    for r, p in enumerate(plans):
        if kin.startswith("flm"):
            ins.append(D.to_dev_c(np.where(masks[r][None, :], full_in, np.nan + 0j)))
        else:
            lay = p.coef_layout if kin == "coef" else p.pix_layout
            ins.append(D.to_dev_c(lay.to_local(full_in)))
    kw = {} if gl is None else {"gl": D.to_dev_f(gl)}
    outs = [_host(o) for o in sim.map(lambda r: getattr(plans[r], method)(ins[r], **kw))]
    nb = full_in.shape[0]
    if kout.startswith("flm"):
        for r, o in enumerate(outs):
            assert not np.any(o[:, ~masks[r]]), f"{method}: rank {r} wrote orders it does not own"
        return np.sum(outs, axis=0)
    n_full = L * (2 * L - 1) if kout == "pix" else plans[0].coef_layout.n_full
    full = np.full((nb, n_full), np.nan + 0j)
    for p, o in zip(plans, outs):
        (p.coef_layout if kout == "coef" else p.pix_layout).scatter_into(full, o)
    assert not np.isnan(full).any(), f"{method}: some rows have no owner"
    return full


def _compare_all(ms, sim, L, U, gl, expect, what):
    """every operation, chain by chain; returns the worst rel-L2"""
    checks = [(0, name, kin, kout, None, name) for name, (kin, kout) in WAVELET_OPS.items()]
    for k, spin in ((1, 0), (2, 2)):
        for fn, (kin, kout) in SHT_OPS.items():
            kin, kout = (f"flm{spin}" if x == "flm" else x for x in (kin, kout))
            for g in (None, gl):
                checks.append((k, fn, kin, kout, g, (spin, fn, g is not None)))
    worst = 0.0
    for k, method, kin, kout, g, key in checks:
        got = _run_sharded(ms, sim, sim.plan_sets[k], method, kin, kout, U[kin], L, g)
        exp = expect[key]
        assert got.shape == exp.shape, (what, key)
        for c in range(got.shape[0]):
            e = rel_l2(got[c], exp[c])
            worst = max(worst, e)
            assert e < TOL, f"{what} {key} chain {c}: rel-L2 {e:.2e}"
    return worst


_EXPECT = {}


def _expected_one_chain(L):
    """unsharded outputs at one chain, computed once per bandlimit (the cases run in order of L)"""
    if L not in _EXPECT:
        _EXPECT.clear()
        from oracle import pxmcmc_ref as R

        ncoefs = R.WaveletTransform(L, B, J_MIN).ncoefs
        U, gl = _basis(L, ncoefs, 1, L)
        _EXPECT[L] = (U, gl) + _unsharded(L, 1, U, gl)
    return _EXPECT[L]


def _sharded_plans(ms, L, world, nb=1):
    return ms.SimulatedRanks(world, lambda r, w: ms.ShardedWaveletPlan(L, B, J_MIN, r, w, nbatch=nb),
                             lambda r, w: ms.ShardedShtPlan(L, 0, r, w, nbatch=nb),
                             lambda r, w: ms.ShardedShtPlan(L, 2, r, w, nbatch=nb))


# ------------------------------------------------------------------ 1. transforms
@pytest.mark.parametrize("L,world", TRANSFORM_CASES, ids=[f"L{L}-w{w}" for L, w in TRANSFORM_CASES])
def test_transforms_sharded_against_unsharded(ms, L, world):
    """the four wavelet operators, the harmonic pair and the four SHTs of spin 0 and 2 with and without a per-degree
    multiplier, sharded over `world` ranks against the unsharded plan, rel-L2 < 1e-13; every operation runs twice, so
    the second call overwrites ring buffers the first one used"""
    U, gl, expect, ncoefs, bl = _expected_one_chain(L)
    assert bl == bandlimits(L)
    sim = _sharded_plans(ms, L, world)
    try:
        assert sim.plans[0].ncoefs == ncoefs
        _compare_all(ms, sim, L, U, gl, expect, f"L={L} world={world}")
        worst = _compare_all(ms, sim, L, U, gl, expect, f"L={L} world={world} (second call)")
    finally:
        _destroy_sim(sim)
    mm = dispatch_mismatches(L, world, 1)
    print(f"\nsharded transforms L={L} world={world}: worst rel-L2 {worst:.2e}"
          + (f"; ring-FFT kernels differ from the unsharded plan at {mm}" if mm else ""))


@pytest.mark.parametrize("L,world", WIDE_CASES, ids=[f"L{L}-w{w}-nb{NB_WIDE}" for L, w in WIDE_CASES])
def test_transforms_sharded_64_chains(ms, L, world):
    """`nbatch = 64` on the sharded plans against the unsharded 64-chain plans, chain by chain, chain scales 1e-6 ... 1"""
    from oracle import pxmcmc_ref as R

    ncoefs = R.WaveletTransform(L, B, J_MIN).ncoefs
    Ub, gl = _basis(L, ncoefs, 3, 7 * L + world)
    a = chain_coefficients(NB_WIDE, 11 * L + world)
    U = {k: a @ u for k, u in Ub.items()}
    expect, _, _ = _unsharded(L, NB_WIDE, U, gl)
    sim = _sharded_plans(ms, L, world, NB_WIDE)
    try:
        worst = _compare_all(ms, sim, L, U, gl, expect, f"L={L} world={world} nb={NB_WIDE}")
    finally:
        _destroy_sim(sim)
    mm = dispatch_mismatches(L, world, NB_WIDE)
    print(f"\nsharded transforms L={L} world={world} nb={NB_WIDE}: worst rel-L2 {worst:.2e}"
          + (f"; ring-FFT kernels differ from the unsharded plan at {mm}" if mm else ""))


# ------------------------------------------------------------------ 2. / 3. the benchmark's weak-lensing chain
WL_L = 512
WL_SEED = 4321
K_ITERS = 5
N_REPLAYS = 4
CHAIN_CASES = [(2, False), (3, True)]  # (world, complex noise): bench.py's chain is (N, False), Philox mode 2


class _Problem:
    """bench.py's config-4 set-up (measure_msharded) with the unsharded operator and sampler next to it"""

    def __init__(self, cplx):
        import bench
        from pxmcmc_b200 import device as D
        from pxmcmc_b200.forward import ForwardOperator
        from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
        from pxmcmc_b200.measurements import WeakLensing
        from pxmcmc_b200.prior import S2_Wavelets_L1
        from pxmcmc_b200.transforms import SphericalWaveletTransform

        L = WL_L
        self.mask, self.ngal = bench.wl_mask(L), np.full((L, 2 * L - 1), 30.0)
        tr = SphericalWaveletTransform(L, B, J_MIN)
        wl = WeakLensing(L, mask=self.mask, ngal=self.ngal)
        rng = np.random.default_rng(11)
        x_true = rng.laplace(size=tr.ncoefs) * 1e-3
        data = np.asarray(wl.forward(tr.inverse(x_true)))
        self.data = data + _crandn(rng, wl.ndata)
        self.sig = 1.0 / np.asarray(wl.inv_cov)
        self.op = ForwardOperator(self.data, self.sig, "synthesis", transform=tr, measurement=wl, nparams=tr.ncoefs)
        # lmda = delta / 2, the benchmark's step
        self.prm = PxMCMCParams(delta=2e-12, lmda=1e-12, mu=1.0, verbosity=0, nsamples=1, nburn=0, ngap=1, track=[],
                                complex=cplx)
        self.reg = S2_Wavelets_L1("synthesis", tr.inverse, tr.inverse_adjoint, self.prm.lmda * self.prm.mu, L=L, B=B,
                                  J_min=J_MIN)
        self.m = MYULA(self.op, self.reg, self.prm)
        self.T = np.asarray(self.reg.T)
        self.Tdev = self.reg._T_args()[0]
        self.X0 = D.to_dev_c(_crandn(rng, 1, tr.ncoefs) * 1e-6)
        self.P0 = D.to_dev_c(self.op.forward(self.X0))
        self.mode = 3 if cplx else 2

    def step(self, X, P, w_re, w_im):
        """one iteration of the unsharded sampler with injected normals"""
        from pxmcmc_b200 import device as D

        g = D.to_dev_c(self.m._gradg_dev(P))
        Xn = D.myula_update_dev(X, None, g, self.Tdev, 0.0, self.prm.delta, self.prm.lmda, w_re=D.to_dev_f(w_re),
                                w_im=None if w_im is None else D.to_dev_f(w_im), noise_mode=1)
        return Xn, D.to_dev_c(self.m._forward_dev(Xn))


class _Sharded:
    """the benchmark's per-rank operator, prior and sampler (MYULA(noise="device", stream0=rank)) on SimulatedRanks"""

    def __init__(self, ms, prob, world):
        from pxmcmc_b200 import device as D
        from pxmcmc_b200.forward import ForwardOperator

        L = WL_L
        self.ms, self.prob, self.world = ms, prob, world
        self.sim = ms.SimulatedRanks(world, lambda r, w: ms.ShardedWaveletPlan(L, B, J_MIN, r, w),
                                     lambda r, w: ms.ShardedShtPlan(L, 0, r, w), lambda r, w: ms.ShardedShtPlan(L, 2, r, w))
        self.tr, self.wl, self.ops, self.regs, self.X0, self.P0 = [], [], [], [], [], []
        for r in range(world):
            t_r = ms.ShardedSphericalWaveletTransform(L, B, J_MIN, r, world, plan=self.sim.plan_sets[0][r])
            w_r = ms.ShardedWeakLensing(L, r, world, mask=prob.mask, ngal=prob.ngal,
                                        plans=(self.sim.plan_sets[1][r], self.sim.plan_sets[2][r]))
            o_r = ForwardOperator(prob.data[w_r.data_index], prob.sig[w_r.data_index], "synthesis", transform=t_r,
                                  measurement=w_r, nparams=t_r.ncoefs)
            g_r = ms.sharded_s2_wavelets_l1(t_r, prob.prm.lmda * prob.prm.mu, L, B, J_MIN)
            assert np.array_equal(np.asarray(g_r.T), prob.T[t_r.coef_layout.index])
            self.tr.append(t_r)
            self.wl.append(w_r)
            self.ops.append(o_r)
            self.regs.append(g_r)
            self.X0.append(D.to_dev_c(t_r.coef_layout.to_local(D.to_host(prob.X0))))
            self.P0.append(D.to_dev_c(D.to_host(prob.P0)[:, w_r.data_index]))
        idx = np.concatenate([t.coef_layout.index for t in self.tr])
        assert np.array_equal(np.sort(idx), np.arange(prob.op.nparams))  # every coefficient has exactly one owner
        assert np.array_equal(np.sort(np.concatenate([w.data_index for w in self.wl])), np.arange(len(prob.data)))

    def samplers(self):
        from pxmcmc_b200.mcmc import MYULA

        return [MYULA(self.ops[r], self.regs[r], self.prob.prm, noise="device", seed=WL_SEED, stream0=r)
                for r in range(self.world)]

    def gather(self, per_rank):
        """full (X, P) host vectors from [(X_r, P_r)]"""
        X = np.zeros(self.prob.op.nparams, dtype=complex)
        P = np.zeros(len(self.prob.data), dtype=complex)
        for r, (x, p) in enumerate(per_rank):
            self.tr[r].coef_layout.scatter_into(X, _host(x).ravel())
            P[self.wl[r].data_index] = _host(p).ravel()
        return X, P

    def noise(self, step):
        """the normals every rank's update draws at `step` (Philox stream = rank, element = local index), as full
        vectors (w_re, w_im or None) and per rank"""
        n = self.prob.op.nparams
        w_re, w_im = np.full(n, np.nan), np.full(n, np.nan)
        per_rank = []
        for r in range(self.world):
            lay = self.tr[r].coef_layout
            re, im = philox_ref.element_normals(self.prob.mode, 1, lay.n_local, WL_SEED, step, stream0=r)
            lay.scatter_into(w_re, re[0])
            lay.scatter_into(w_im, im[0])
            per_rank.append(re[0])
        assert not np.isnan(w_re).any()
        return w_re, (w_im if self.prob.mode == 3 else None), per_rank


@pytest.fixture(scope="module", params=CHAIN_CASES, ids=[f"w{w}-{'complex' if c else 'real'}-noise" for w, c in CHAIN_CASES])
def wl_chain(ms, request):
    """(problem, sharded set-up, eager sharded chain: [(X_r, P_r) per rank] after each of K iterations enqueued back to
    back, the samplers that ran it) for one (world, complex noise)"""
    import torch

    world, cplx = request.param
    prob = _Problem(cplx)
    sh = _Sharded(ms, prob, world)
    samplers = sh.samplers()
    torch.cuda.synchronize()

    def chain(r):
        X, P, out = sh.X0[r], sh.P0[r], []
        for _ in range(K_ITERS):
            X, P = samplers[r].iterate(X, P)
            out.append((X.clone(), P.clone()))
        return out

    try:
        per_rank = sh.sim.map(chain)
        yield prob, sh, [[per_rank[r][k] for r in range(world)] for k in range(K_ITERS)], samplers
    finally:
        _destroy_sim(sh.sim)


def _check_iteration(prob, sh, got, Xn, Pn, what):
    """sharded (X, P) per rank against the unsharded ones: state / predictions, prox support, sign pattern, log-pi parts"""
    Xs, Ps = sh.gather(got)
    from pxmcmc_b200 import device as D

    xn, pn = D.to_host(Xn).ravel(), D.to_host(Pn).ravel()
    ex, ep = rel_l2(Xs, xn), rel_l2(Ps, pn)
    assert ex < 1e-12 and ep < 1e-12, f"{what}: rel-L2 state {ex:.2e}, predictions {ep:.2e}"
    assert np.array_equal(np.abs(Xs) > prob.T, np.abs(xn) > prob.T), f"{what}: prox support"
    assert np.array_equal(np.sign(Xs.real), np.sign(xn.real)) and np.array_equal(np.sign(Xs.imag), np.sign(xn.imag)), \
        f"{what}: sign pattern"
    _, l2, pr = prob.m._logpi_dev(Xn, Pn)
    parts = []
    for r in range(sh.world):
        from pxmcmc_b200.mcmc import MYULA

        mr = MYULA(sh.ops[r], sh.regs[r], prob.prm)
        parts.append(mr._logpi_dev(got[r][0], got[r][1]))
    sl2, spr = sum(p[1][0] for p in parts), sum(p[2][0] for p in parts)
    assert abs(sl2 - l2[0]) <= 1e-11 * abs(l2[0]), f"{what}: L2 {sl2} vs {l2[0]}"
    assert abs(spr - pr[0]) <= 1e-11 * abs(pr[0]), f"{what}: prior {spr} vs {pr[0]}"
    return max(ex, ep)


def _check_device_noise(sh, per_rank, w_im):
    """the normals each rank's sampler draws on the device at step 1, from the update of a zero state with a zero
    gradient (X' = sqrt(2 delta) w), against the restatement of Philox stream `rank`; two ranks' draws must differ"""
    import torch

    from pxmcmc_b200 import device as D

    prob, draws = sh.prob, []
    for r, m in enumerate(sh.samplers()):
        zero = torch.zeros_like(sh.X0[r])
        w = D.to_host(m._propose_dev(zero, None, zero))[0] / np.sqrt(2 * prob.prm.delta)
        assert m._step_counter == 1
        exp = per_rank[r] if w_im is None else per_rank[r] + 1j * w_im[sh.tr[r].coef_layout.index]
        assert rel_l2(w, exp) < 1e-13, f"rank {r}: device noise is not Philox stream {r}"
        if w_im is None:
            assert not np.any(w.imag), f"rank {r}: real noise expected"
        draws.append(w)
    n = min(len(w) for w in draws)
    for r in range(1, sh.world):
        assert not np.array_equal(draws[0][:n], draws[r][:n]), f"ranks 0 and {r} draw the same normals on the device"


def test_myula_iterations_back_to_back(ms, wl_chain):
    """K = 5 `MYULA.iterate` calls per rank enqueued with no host synchronisation, Philox noise on the device with
    stream0 = rank, against the unsharded sampler stepped with the restated normals: state and predictions rel-L2
    < 1e-12, identical prox support and sign pattern, per-rank log-pi parts adding up to 1e-11; then one iteration of
    the literal composition (fuse_harmonic = False on both operators).  At the benchmark's step the thresholds
    (lmda mu w, about 1e-12) are far below |X| (about 1e-6), so every coefficient is in the prox support and the sign
    pattern is the check that bites.  Each rank's device noise is also read back directly: the update of a zero
    state with a zero gradient is sqrt(2 delta) w, which must be the restated normals of Philox stream `rank`."""
    prob, sh, eager, samplers = wl_chain
    assert prob.op._fused() and all(o._fused() for o in sh.ops)
    assert all(m.noise == "device" and m.complex == (prob.mode == 3) for m in samplers)
    # MYULA._propose_dev: every eager iterate advances _step_counter first, so iteration k draws step k
    assert all(m._step_counter == K_ITERS for m in samplers)
    X, P = prob.X0, prob.P0
    worst = 0.0
    for k in range(1, K_ITERS + 1):
        w_re, w_im, per_rank = sh.noise(k)
        if k == 1:
            _check_device_noise(sh, per_rank, w_im)
        X, P = prob.step(X, P, w_re, w_im)
        worst = max(worst, _check_iteration(prob, sh, eager[k - 1], X, P, f"iteration {k}"))
    # the literal composition: the full-L SHT pair between Psi and Phi is executed instead of skipped
    for o in sh.ops + [prob.op]:
        o.fuse_harmonic = False
    try:
        assert not prob.op._fused() and not any(o._fused() for o in sh.ops)
        last = eager[-1]
        got = sh.sim.map(lambda r: samplers[r].iterate(last[r][0], last[r][1]))
        w_re, w_im, _ = sh.noise(K_ITERS + 1)
        Xl, Pl = prob.step(X, P, w_re, w_im)
        worst_lit = _check_iteration(prob, sh, got, Xl, Pl, "literal composition")
    finally:
        for o in sh.ops + [prob.op]:
            o.fuse_harmonic = True
    print(f"\nMYULA L={WL_L} world={sh.world} mode {prob.mode}: worst rel-L2 over {K_ITERS} back-to-back iterations "
          f"{worst:.2e}, literal composition {worst_lit:.2e}")


def test_graph_replay_across_ranks(ms, wl_chain):
    """`GraphedChain`'s capture block done rank by rank: warm-up of every rank in one `map`, the device step counters
    set, each rank's iteration captured on its own stream (capture executes nothing), then every graph replayed
    4 times in one `map`.  `GraphedChain` itself cannot be used here:
    `torch.cuda.graph` synchronises the device when it starts a capture, which on one GPU would wait for rank 0's
    warm-up, and that waits in a barrier for ranks not enqueued yet (one process per GPU does not have this problem:
    test_two_processes_myula_L512).  The replayed chain equals the eager one to 1e-14, every barrier met its peers."""
    import torch

    prob, sh, eager, _ = wl_chain
    world = sh.world
    samplers = sh.samplers()
    X = [x.clone() for x in sh.X0]
    P = [p.clone() for p in sh.P0]
    for m in samplers:
        m._dstep = torch.full((1,), m._step_counter + 1, dtype=torch.int64, device=X[0].device)
    try:
        def warm(r):
            x, p = X[r].clone(), P[r].clone()
            for _ in range(2):
                x, p = samplers[r].iterate(x, p)
        sh.sim.map(warm)
        for m in samplers:
            m._dstep.fill_(m._step_counter + 1)  # the warm-up is not part of the chain
        graphs = []
        for r in range(world):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=sh.sim.streams[r]):
                samplers[r].iterate(X[r], P[r], out=(X[r], P[r]))
            graphs.append(g)

        def replay(r):
            for _ in range(N_REPLAYS):
                graphs[r].replay()
        sh.sim.map(replay)
        assert all(int(m._dstep.item()) == N_REPLAYS + 1 for m in samplers)
        assert all(p.barrier_ok() for plans in sh.sim.plan_sets for p in plans)
        Xg, Pg = sh.gather(list(zip(X, P)))
        Xe, Pe = sh.gather(eager[N_REPLAYS - 1])
        ex, ep = rel_l2(Xg, Xe), rel_l2(Pg, Pe)
        print(f"\ngraph replay L={WL_L} world={world}: rel-L2 to the eager chain after {N_REPLAYS} replays: "
              f"state {ex:.2e}, predictions {ep:.2e}")
        assert ex <= 1e-14 and ep <= 1e-14
        del graphs
    finally:
        for m in samplers:
            m._dstep = None


# ------------------------------------------------------------------ 4. one process per GPU
def test_two_processes_myula_L512():
    """`scripts/msharded_check.py --iterate 5` on two GPUs: the sampler's own iteration over CUDA IPC and NVLink, eager
    and through `MYULA.capture` / `GraphedChain`, against the unsharded chain with the restated noise"""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "scripts", "msharded_check.py"), "--L", "512", "--B", "2",
           "--iterate", "5"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MSHARDED OK" in r.stdout
