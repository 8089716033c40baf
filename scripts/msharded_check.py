#!/usr/bin/env python
"""One process per GPU (torchrun): parity and timing of the m-sharded transforms.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node=2 --master-addr 127.0.0.1 \
        scripts/msharded_check.py --L 136 --B 2 [--bench]

Every rank also owns an unsharded plan of the same transform, so the expected
result is computed on the spot; rank 0 prints `MSHARDED OK` when every rank agrees
to 1e-12 relative L2, and one JSON line of timings with --bench.

--iterate K: also K iterations of bench.py's config-4 chain (weak lensing, `MYULA(noise="device", stream0=rank)`),
eagerly and replayed through `MYULA.capture`, against the unsharded sampler on every rank stepped with the same
Philox normals restated on the host (oracle/philox_ref.py): state and predictions to 1e-12 relative L2, the
all-reduced L2 and prior terms to 1e-11.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, default=136)
    ap.add_argument("--B", type=float, default=2.0)
    ap.add_argument("--J_min", type=int, default=2)
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--iterate", type=int, default=0)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    os.environ.pop("NCCL_DEBUG", None)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from pxmcmc_b200 import device as D
    from pxmcmc_b200 import msharded as ms

    L, B, J = args.L, args.B, args.J_min
    ex = ms.ProcessGroupExchange()
    wp = ms.ShardedWaveletPlan(L, B, J, rank, world, exchange=ex)
    s0 = ms.ShardedShtPlan(L, 0, rank, world, exchange=ex)
    s2 = ms.ShardedShtPlan(L, 2, rank, world, exchange=ex)
    whole_w = D.WaveletPlan.get(L, B, J, 1)
    rng = np.random.default_rng(99)  # same stream on every rank
    coef = rng.standard_normal(wp.ncoefs) + 1j * rng.standard_normal(wp.ncoefs)
    pix = rng.standard_normal(L * (2 * L - 1)) + 1j * rng.standard_normal(L * (2 * L - 1))
    flm = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    flm[:4] = 0
    worst = 0.0

    def rel(a, b):
        return float(np.linalg.norm(a - b) / np.linalg.norm(b))

    checks = [("synthesis", coef, wp.coef_layout, wp.pix_layout), ("synthesis_adjoint", pix, wp.pix_layout, wp.coef_layout),
              ("analysis", pix, wp.pix_layout, wp.coef_layout), ("analysis_adjoint", coef, wp.coef_layout, wp.pix_layout)]
    for name, full_in, lin, lout in checks:
        expect = getattr(whole_w, name)(D.to_dev_c(full_in)).cpu().numpy()
        for _ in range(2):
            got = getattr(wp, name)(D.to_dev_c(lin.to_local(full_in))).cpu().numpy()
        e = rel(got, lout.to_local(expect)) if got.size else 0.0
        worst = max(worst, e)
        if rank == 0:
            print(f"wavelet {name}: rank0 rel-L2 {e:.2e}", flush=True)
    mask = ms.flm_owner_mask(L, rank, world)
    for spin, sp in ((0, s0), (2, s2)):
        whole = D.ShtPlan.get(L, spin, 1)
        for name, harm_in in (("inverse", True), ("forward_adjoint", True), ("forward", False), ("inverse_adjoint", False)):
            expect = getattr(whole, name)(D.to_dev_c(flm if harm_in else pix)).cpu().numpy()
            if harm_in:
                got = getattr(sp, name)(D.to_dev_c(np.where(mask, flm, 0))).cpu().numpy()
                e = rel(got, sp.pix_layout.to_local(expect)) if got.size else 0.0
            else:
                got = getattr(sp, name)(D.to_dev_c(sp.pix_layout.to_local(pix))).cpu().numpy()
                e = rel(got, np.where(mask, expect, 0))
            worst = max(worst, e)
            if rank == 0:
                print(f"sht spin {spin} {name}: rank0 rel-L2 {e:.2e}", flush=True)
    if args.iterate:
        worst = max(worst, iterate_check(args.iterate, rank, world, wp, s0, s2, rel))
    ok = wp.barrier_ok() and s0.barrier_ok() and s2.barrier_ok() and worst < 1e-12
    t = torch.tensor([0.0 if ok else 1.0, worst], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(f"worst rel-L2 over ranks {t[1].item():.2e}", flush=True)
        print("MSHARDED OK" if t[0].item() == 0.0 else "MSHARDED FAILED", flush=True)

    if args.bench:
        xc = D.to_dev_c(wp.coef_layout.to_local(coef))
        xp = D.to_dev_c(wp.pix_layout.to_local(pix))
        res = {"L": L, "B": B, "world": world}
        for name, x in (("synthesis", xc), ("synthesis_adjoint", xp)):
            for _ in range(5):
                getattr(wp, name)(x)
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                getattr(wp, name)(x)
            e1.record()
            torch.cuda.synchronize()
            tt = torch.tensor([e0.elapsed_time(e1) / args.iters], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            res[f"sharded_{name}_ms"] = tt.item()
            xf = D.to_dev_c(coef if name == "synthesis" else pix)
            for _ in range(3):
                getattr(whole_w, name)(xf)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.iters):
                getattr(whole_w, name)(xf)
            e1.record()
            torch.cuda.synchronize()
            res[f"single_gpu_{name}_ms"] = e0.elapsed_time(e1) / args.iters
        if rank == 0:
            print(json.dumps(res), flush=True)
            if args.out:
                with open(args.out, "w") as f:
                    json.dump(res, f)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if t[0].item() == 0.0 else 1)


def iterate_check(K, rank, world, wp, s0, s2, rel):
    """worst relative error of K iterations of the sharded chain, eager and graphed, against the unsharded one"""
    from bench import wl_mask
    from oracle import philox_ref
    from pxmcmc_b200 import device as D
    from pxmcmc_b200 import msharded as ms
    from pxmcmc_b200.forward import ForwardOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.measurements import WeakLensing
    from pxmcmc_b200.prior import S2_Wavelets_L1
    from pxmcmc_b200.transforms import SphericalWaveletTransform

    L, B, J, seed = wp.L, wp.B, wp.J_min, 4321
    mask, ngal = wl_mask(L), np.full((L, 2 * L - 1), 30.0)
    # the unsharded problem, the same on every rank
    tr = SphericalWaveletTransform(L, B, J)
    wl = WeakLensing(L, mask=mask, ngal=ngal)
    rng = np.random.default_rng(11)
    data = np.asarray(wl.forward(tr.inverse(rng.laplace(size=tr.ncoefs) * 1e-3)))
    data = data + rng.standard_normal(wl.ndata) + 1j * rng.standard_normal(wl.ndata)
    sig = 1.0 / np.asarray(wl.inv_cov)
    op = ForwardOperator(data, sig, "synthesis", transform=tr, measurement=wl, nparams=tr.ncoefs)
    prm = PxMCMCParams(delta=2e-12, lmda=1e-12, mu=1.0, verbosity=0, nsamples=1, nburn=0, ngap=1, track=[])
    reg = S2_Wavelets_L1("synthesis", tr.inverse, tr.inverse_adjoint, prm.lmda * prm.mu, L=L, B=B, J_min=J)
    full = MYULA(op, reg, prm)
    X0 = (rng.standard_normal((1, tr.ncoefs)) + 1j * rng.standard_normal((1, tr.ncoefs))) * 1e-6
    layouts = [ms.MapLayout(wp.bandlimits, range(1, len(wp.bandlimits) + 1), r, world) for r in range(world)]
    X, P = D.to_dev_c(X0), D.to_dev_c(op.forward(D.to_dev_c(X0)))
    expect = []
    for k in range(1, K + 1):
        # rank r's update draws Philox stream r (mode 2: real noise on the complex state) at its local element index
        w = np.zeros(tr.ncoefs)
        for r, lay in enumerate(layouts):
            lay.scatter_into(w, philox_ref.element_normals(2, 1, lay.n_local, seed, k, stream0=r)[0][0])
        g = D.to_dev_c(full._gradg_dev(P))
        X = D.myula_update_dev(X, None, g, reg._T_args()[0], 0.0, prm.delta, prm.lmda, w_re=D.to_dev_f(w), noise_mode=1)
        P = D.to_dev_c(full._forward_dev(X))
        _, l2, pr = full._logpi_dev(X, P)
        expect.append((D.to_host(X), D.to_host(P), l2[0], pr[0]))
    # this rank's share, with the scalar reductions over the process group
    t_r = ms.ShardedSphericalWaveletTransform(L, B, J, rank, world, plan=wp)
    w_r = ms.ShardedWeakLensing(L, rank, world, mask=mask, ngal=ngal, plans=(s0, s2))
    o_r = ForwardOperator(data[w_r.data_index], sig[w_r.data_index], "synthesis", transform=t_r, measurement=w_r,
                          nparams=t_r.ncoefs)
    o_r._pxm_allreduce = ms.allreduce_sum()
    assert o_r._fused() and op._fused()
    g_r = ms.sharded_s2_wavelets_l1(t_r, prm.lmda * prm.mu, L, B, J)
    idx, didx = t_r.coef_layout.index, w_r.data_index
    Xl0 = D.to_dev_c(X0[:, idx])
    Pl0 = D.to_dev_c(D.to_host(op.forward(D.to_dev_c(X0)))[:, didx])
    worst = 0.0

    def check(k, m, Xl, Pl, what):
        xe, pe, l2, pr = expect[k - 1]
        e = max(rel(D.to_host(Xl).ravel(), xe[0, idx]), rel(D.to_host(Pl).ravel(), pe[0, didx]))
        _, l2s, prs = m._logpi_dev(Xl, Pl)
        e_lp = max(abs(l2s[0] - l2) / abs(l2), abs(prs[0] - pr) / abs(pr))
        if rank == 0:
            print(f"{what} iteration {k}: rank0 rel-L2 {e:.2e}, log-pi terms {e_lp:.2e}", flush=True)
        return e if e_lp <= 1e-11 else max(e, 1.0)

    m = MYULA(o_r, g_r, prm, noise="device", seed=seed, stream0=rank)
    Xl, Pl = Xl0, Pl0
    for k in range(1, K + 1):
        Xl, Pl = m.iterate(Xl, Pl)
        worst = max(worst, check(k, m, Xl, Pl, "eager"))
    m = MYULA(o_r, g_r, prm, noise="device", seed=seed, stream0=rank)
    chain = m.capture(Xl0, Pl0, iterations=1)
    for k in range(1, K + 1):
        chain.step()
        Xl, Pl = chain.state()
        worst = max(worst, check(k, m, Xl, Pl, "graphed"))
    chain.release()
    return worst


if __name__ == "__main__":
    main()
