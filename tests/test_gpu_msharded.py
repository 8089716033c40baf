"""GPU tests of the m-sharded transforms (SURVEY.md 8e-2).

* `SimulatedRanks`: all ranks of a sharded plan live in ONE process on ONE GPU (one
  stream per rank) -- the same kernels, peer-pointer tables, push/pull contractions
  and flag barrier as the multi-process path, so the driver's single-GPU
  `pytest -m gpu` covers it.  Reference values: the CPU oracle at small L, the
  unsharded plan (itself pinned to the oracle/fixtures in test_gpu_parity.py) at
  bandlimits with several 64-ring blocks.
* `test_two_processes_*`: real one-process-per-GPU run over CUDA IPC + NVLink,
  skipped when fewer than two GPUs are visible.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-10  # relative L2, FP64 (BASELINE.json north_star)


@pytest.fixture(scope="module")
def ms():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pxmcmc_b200 import msharded

    return msharded


def _dev(x):
    from pxmcmc_b200 import device as D

    return D.to_dev_c(x)


def _host(t):
    return t.detach().cpu().numpy()


def _rand_c(rng, n):
    return rng.standard_normal(n) + 1j * rng.standard_normal(n)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_wavelet_small_L_against_oracle(ms, world):
    L, B, J = 20, 2.0, 1
    rng = np.random.default_rng(5)
    sim = ms.SimulatedRanks(world, lambda r, w: ms.ShardedWaveletPlan(L, B, J, r, w))
    p0 = sim.plans[0]
    coef = _rand_c(rng, p0.ncoefs)
    pix = _rand_c(rng, L * (2 * L - 1))
    from oracle import pxmcmc_ref as R

    t = R.WaveletTransform(L, B, J)
    expect = {"synthesis": t.inverse(coef), "synthesis_adjoint": t.inverse_adjoint(pix),
              "analysis": t.forward(pix), "analysis_adjoint": t.forward_adjoint(coef)}
    for name, full_in, in_lay, out_lay in [
        ("synthesis", coef, "coef_layout", "pix_layout"),
        ("synthesis_adjoint", pix, "pix_layout", "coef_layout"),
        ("analysis", pix, "pix_layout", "coef_layout"),
        ("analysis_adjoint", coef, "coef_layout", "pix_layout"),
    ]:
        ins = [_dev(getattr(p, in_lay).to_local(full_in)) for p in sim.plans]
        outs = sim.run(name, ins)
        full = np.zeros(getattr(p0, out_lay).n_full, dtype=complex)
        for p, o in zip(sim.plans, outs):
            getattr(p, out_lay).scatter_into(full, _host(o))
        assert rel_l2(full, expect[name]) < TOL, name


@pytest.mark.parametrize("world,L,B", [(2, 136, 2.0), (4, 200, 1.7), (8, 136, 2.0)])
def test_wavelet_multiblock_against_unsharded(ms, world, L, B):
    from pxmcmc_b200 import device as D

    J = 2
    rng = np.random.default_rng(11)
    whole = D.WaveletPlan.get(L, B, J, 1)
    sim = ms.SimulatedRanks(world, lambda r, w: ms.ShardedWaveletPlan(L, B, J, r, w))
    p0 = sim.plans[0]
    assert p0.ncoefs == whole.ncoefs
    # every rank owns 1/world of the tables (up to the snake's granularity)
    tb = [p.table_bytes for p in sim.plans]
    assert max(tb) < 0.75 * whole.table_bytes
    coef = _rand_c(rng, p0.ncoefs)
    pix = _rand_c(rng, L * (2 * L - 1))
    for name, full_in, in_lay, out_lay in [
        ("synthesis", coef, "coef_layout", "pix_layout"),
        ("synthesis_adjoint", pix, "pix_layout", "coef_layout"),
        ("analysis", pix, "pix_layout", "coef_layout"),
        ("analysis_adjoint", coef, "coef_layout", "pix_layout"),
    ]:
        expect = _host(getattr(whole, name)(_dev(full_in)))
        # twice: the second call checks that the ring buffers are safely reused across calls
        for _ in range(2):
            ins = [_dev(getattr(p, in_lay).to_local(full_in)) for p in sim.plans]
            outs = sim.run(name, ins)
        full = np.zeros(getattr(p0, out_lay).n_full, dtype=complex)
        for p, o in zip(sim.plans, outs):
            getattr(p, out_lay).scatter_into(full, _host(o))
        assert rel_l2(full, expect) < 1e-13, name


@pytest.mark.parametrize("spin", [0, 2])
@pytest.mark.parametrize("world,L", [(2, 24), (4, 150)])
def test_sht_sharded(ms, spin, world, L):
    from oracle import ssht_ref
    from pxmcmc_b200 import device as D

    rng = np.random.default_rng(3)
    sim = ms.SimulatedRanks(world, lambda r, w: ms.ShardedShtPlan(L, spin, r, w))
    flm = _rand_c(rng, L * L)
    for el in range(abs(spin)):
        flm[el * el:(el + 1) * (el + 1)] = 0
    f = _rand_c(rng, L * (2 * L - 1))
    whole = D.ShtPlan.get(L, spin, 1)
    gl = D.to_dev_f(rng.standard_normal(L))
    masks = [ms.flm_owner_mask(L, r, world) for r in range(world)]
    assert np.array_equal(np.sum(masks, axis=0), np.ones(L * L))  # every order has exactly one owner
    for name, harmonic_in in [("inverse", True), ("forward_adjoint", True), ("forward", False), ("inverse_adjoint", False)]:
        for g in (None, gl):
            if L <= 32 and g is None:
                fn = getattr(ssht_ref, name)
                expect = np.asarray(fn(flm if harmonic_in else f.reshape(L, 2 * L - 1), L, spin)).ravel()
                tol = TOL
            else:
                expect = _host(getattr(whole, name)(_dev(flm if harmonic_in else f), gl=g))
                tol = 1e-13
            if harmonic_in:
                # a rank is only required to hold its own orders: poison the rest
                ins = [_dev(np.where(mk, flm, np.nan + 0j)) for mk in masks]
                outs = sim.run(name, ins, gl=g)
                full = np.zeros(L * (2 * L - 1), dtype=complex)
                for p, o in zip(sim.plans, outs):
                    p.pix_layout.scatter_into(full, _host(o))
            else:
                ins = [_dev(p.pix_layout.to_local(f)) for p in sim.plans]
                outs = [_host(o) for o in sim.run(name, ins, gl=g)]
                for mk, o in zip(masks, outs):
                    assert not np.any(o[~mk])  # orders of other ranks read as zero
                full = np.sum(outs, axis=0)
            assert rel_l2(full, expect) < tol, (name, g is not None)


def test_two_processes_over_nvlink():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "scripts", "msharded_check.py"), "--L", "136", "--B", "2"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MSHARDED OK" in r.stdout


@pytest.mark.parametrize("world", [2, 4])
def test_weaklensing_myula_iteration_sharded(ms, world):
    """config 4 of BASELINE.json in miniature: one MYULA iteration of the spin-2 weak-lensing
    operator with an S2_Wavelets_L1 prior, sharded over `world` ranks, against the unsharded
    sampler with the same injected noise (which test_gpu_parity.py pins to the reference fixture)."""
    import torch

    from pxmcmc_b200 import device as D
    from pxmcmc_b200.forward import ForwardOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.measurements import WeakLensing
    from pxmcmc_b200.prior import S2_Wavelets_L1
    from pxmcmc_b200.transforms import SphericalWaveletTransform

    L, B, J = 72, 2.0, 2
    rng = np.random.default_rng(21)
    mask = rng.random((L, 2 * L - 1)) < 0.6
    ngal = np.full((L, 2 * L - 1), 30.0)
    wl = WeakLensing(L, mask=mask, ngal=ngal)
    tr = SphericalWaveletTransform(L, B, J)
    data = _rand_c(rng, wl.ndata)
    sig = 1.0 / wl.inv_cov
    op = ForwardOperator(data, sig, "synthesis", transform=tr, measurement=wl, nparams=tr.ncoefs)
    prm = PxMCMCParams(delta=1e-3, lmda=2e-3, mu=1.0, nsamples=1, verbosity=0, track=[])
    reg = S2_Wavelets_L1("synthesis", tr.inverse, tr.inverse_adjoint, prm.lmda * prm.mu * 50, L=L, B=B, J_min=J)
    m = MYULA(op, reg, prm)
    X = rng.laplace(size=tr.ncoefs) + 0j
    P = op.forward(X)
    w = rng.standard_normal(tr.ncoefs)
    Tfull = np.asarray(reg.T)
    gradg = op.calc_gradg(P)
    Xn = D.to_host(D.myula_update_dev(D.to_dev_c(X), None, D.to_dev_c(gradg), D.to_dev_f(Tfull), 0.0, prm.delta, prm.lmda,
                                      w_re=D.to_dev_f(w), noise_mode=1))
    Pn = op.forward(Xn)
    lp, l2, pr = m._logpi_dev(m._state(Xn), m._state(Pn))

    sim = ms.SimulatedRanks(world, lambda r, ws: ms.ShardedWaveletPlan(L, B, J, r, ws),
                            lambda r, ws: ms.ShardedShtPlan(L, 0, r, ws), lambda r, ws: ms.ShardedShtPlan(L, 2, r, ws))
    ops, regs, Xl, Pl, wl_r = [], [], [], [], []
    for r in range(world):
        t_r = ms.ShardedSphericalWaveletTransform(L, B, J, r, world, plan=sim.plan_sets[0][r])
        w_r = ms.ShardedWeakLensing(L, r, world, mask=mask, ngal=ngal, plans=(sim.plan_sets[1][r], sim.plan_sets[2][r]))
        o_r = ForwardOperator(data[w_r.data_index], sig[w_r.data_index], "synthesis", transform=t_r, measurement=w_r,
                              nparams=t_r.ncoefs)
        o_r._upload()
        g_r = ms.sharded_s2_wavelets_l1(t_r, prm.lmda * prm.mu * 50, L, B, J)
        assert np.array_equal(np.asarray(g_r.T), Tfull[t_r.coef_layout.index])
        ops.append(o_r)
        regs.append(g_r)
        wl_r.append(w_r)
        Xl.append(D.to_dev_c(t_r.coef_layout.to_local(X)))
        Pl.append(D.to_dev_c(P[w_r.data_index]))
    assert sum(w_r.ndata for w_r in wl_r) == wl.ndata
    Tl = [g._T_args()[0] for g in regs]
    noise = [D.to_dev_f(ops[r].transform.coef_layout.to_local(w)) for r in range(world)]
    torch.cuda.synchronize()

    def iteration(r):
        g = ops[r].calc_gradg(Pl[r])
        xn = D.myula_update_dev(Xl[r], None, g, Tl[r], 0.0, prm.delta, prm.lmda, w_re=noise[r], noise_mode=1)
        return xn, ops[r].forward(xn)

    outs = sim.map(iteration)
    Xs, Ps = np.zeros_like(Xn), np.zeros_like(Pn)
    for r, (xn, pn) in enumerate(outs):
        ops[r].transform.coef_layout.scatter_into(Xs, _host(xn))
        Ps[wl_r[r].data_index] = _host(pn)
    assert rel_l2(Xs, Xn) < 1e-12 and rel_l2(Ps, Pn) < 1e-12
    # prox support / sign pattern identical (north_star)
    assert np.array_equal(Xs == 0, Xn == 0) and np.array_equal(np.sign(Xs.real), np.sign(Xn.real))
    # log posterior: partial sums per rank add up to the unsharded value
    parts = []
    for r in range(world):
        mr = MYULA(ops[r], regs[r], prm)
        parts.append(mr._logpi_dev(mr._state(outs[r][0]), mr._state(outs[r][1])))
    assert abs(sum(p[1][0] for p in parts) - l2[0]) <= 1e-11 * abs(l2[0])
    assert abs(sum(p[2][0] for p in parts) - pr[0]) <= 1e-11 * abs(pr[0])
