"""Cost of the MAP estimate at the operators of configs 1, 3, 4 and 5 (all with a real, positive inverse covariance):
`ForwardOperator.lipschitz()` (wall time, ARPACK's matrix-vector products, and what the host <-> device copies of those
products and the device operator cost on their own), FISTA milliseconds per iteration for 1 and 64 chains (graph
replays), and the iterations `map_estimate` takes to tol = 1e-8.  Prints one JSON object with the card's name and power
limit; `--out FILE` also writes it there.

    python scripts/map_timing.py [--out FILE] [--configs 1,3,4,5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def events_ms(fn, n, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def wl_mask(L):
    """bench.py's config-4 mask"""
    th = (2 * np.arange(L) + 1) * np.pi / (2 * L - 1)
    ph = 2 * np.pi * np.arange(2 * L - 1) / (2 * L - 1)
    T, P = np.meshgrid(th, ph, indexing="ij")
    y, z = np.sin(T) * np.sin(P), np.cos(T)
    a = np.radians(62.87)
    z2 = -np.sin(a) * y + np.cos(a) * z
    mask = np.ones((L, 2 * L - 1), dtype=bool)
    mask[np.abs(np.degrees(np.arcsin(np.clip(z, -1, 1)))) < 10] = False
    mask[np.abs(np.degrees(np.arcsin(np.clip(z2, -1, 1)))) < 10] = False
    return mask


def make(config, nchains):
    """(sampler, description) of a config's operator and prior (MYULA; lmda = 5e-7, mu = 1)"""
    from pxmcmc_b200 import measurements, paths, transforms
    from pxmcmc_b200.forward import ForwardOperator, PathIntegralOperator, SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1, S2_Wavelets_L1_Power_Weights

    lmda = 5e-7
    prm = PxMCMCParams(lmda=lmda, mu=1.0, verbosity=0, nsamples=1, track=[])
    rng = np.random.default_rng(7)
    if config in (1, 5):
        L, B = (32, 1.5) if config == 1 else (256, 1.5)
        data = rng.standard_normal(L * (2 * L - 1))
        op = SphericalWaveletTransformOperator(data, 1.0, "synthesis", L, B, 2, nchains=nchains)
        reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, lmda, L=L, B=B, J_min=2)
        desc = f"wavelet synthesis + identity, L = {L}, B = {B}, scalar sigma (Gram form)"
    elif config == 3:
        L, B = 128, 2
        z = rng.uniform(-1, 1, size=(10000, 2))
        lon = rng.uniform(-180, 180, size=(10000, 2))
        lat = np.degrees(np.arcsin(z))
        A = paths.get_path_matrix(np.stack([lat[:, 0], lon[:, 0]], 1), np.stack([lat[:, 1], lon[:, 1]], 1), L)
        y = A @ rng.standard_normal(A.shape[1]) + 0.05 * rng.standard_normal(A.shape[0])
        op = PathIntegralOperator(A, y, np.full(A.shape[0], 0.05), "synthesis", L, B, 2, nchains=nchains)
        reg = S2_Wavelets_L1_Power_Weights("synthesis", op.transform.inverse, op.transform.inverse_adjoint, lmda, L=L,
                                           B=B, J_min=2, eta=1)
        desc = "10^4 great-circle paths (CSR), L = 128, B = 2"
    else:
        L, B = 512, 2.0
        wl = measurements.WeakLensing(L, mask=wl_mask(L), ngal=np.full((L, 2 * L - 1), 30.0))
        tr = transforms.SphericalWaveletTransform(L, B, 2, nchains=nchains)
        data = rng.standard_normal(wl.ndata) + 1j * rng.standard_normal(wl.ndata)
        op = ForwardOperator(data, (1.0 / wl.inv_cov).astype(complex), "synthesis", transform=tr, measurement=wl,
                             nparams=tr.ncoefs)
        reg = S2_Wavelets_L1("synthesis", tr.inverse, tr.inverse_adjoint, lmda, L=L, B=B, J_min=2)
        desc = "weak lensing (spin 2, masked, ngal = 30) behind a wavelet synthesis, L = 512, B = 2, sigma complex"
    return MYULA(op, reg, prm, nchains=nchains), desc


def lipschitz_cost(m):
    from pxmcmc_b200 import device as D

    op = m.forward
    t0 = time.perf_counter()
    lam = op.lipschitz()
    total_ms = (time.perf_counter() - t0) * 1e3
    nmv = op._lipschitz_cache[3]
    n = op.nparams
    v = np.random.default_rng(0).standard_normal(n).astype(np.complex128)
    z = op._zero_data()
    xd = D.to_dev_c(v).reshape(1, n)

    def copies():
        D.to_host(D.to_dev_c(v))

    def host_clock(fn, reps):
        fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3 / reps

    copy_ms = host_clock(copies, 20)
    apply_ms = events_ms(lambda: z._normal_apply(xd), 20)
    return {"lipschitz": lam, "wall_ms": total_ms, "matvecs": nmv, "copy_ms_per_matvec": copy_ms,
            "device_apply_ms_per_matvec": apply_ms, "copy_share": copy_ms * nmv / total_ms,
            "device_share": apply_ms * nmv / total_ms}


def fista_ms(m, iters):
    """ms per iteration of `map_estimate(tol = 0)` over `iters` iterations (graph replays), the capture excluded by
    differencing two lengths"""
    n = m.forward.nparams
    x0 = np.random.default_rng(1).laplace(size=(m.nchains, n) if m.nchains > 1 else n) * 1e-3
    m.map_estimate(x0, tol=0.0, maxiter=2 * m._FISTA_BLOCK)  # warm: lipschitz cached, tables, pools
    walls = []
    for k in (iters, 2 * iters):
        torch.cuda.synchronize()
        t = time.perf_counter()
        m.map_estimate(x0, tol=0.0, maxiter=k)
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t)
    return (walls[1] - walls[0]) * 1e3 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--configs", default="1,3,4,5")
    ap.add_argument("--maxiter", type=int, default=100_000, help="cap of the run to tol = 1e-8 (config 4: a fifth of it)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(), "method": "lipschitz: host clock around the call; copies: host clock around one vector's "
           "round trip; device operator and FISTA: CUDA events / host clock around work ending in a synchronise"}
    for c in [int(s) for s in args.configs.split(",")]:
        r = {}
        m, r["operator"] = make(c, 1)
        r["nparams"] = int(m.forward.nparams)
        r["lipschitz"] = lipschitz_cost(m)
        iters = 500 if c in (1, 3) else 100
        r["fista_ms_per_iteration_1_chain"] = fista_ms(m, iters)
        n = m.forward.nparams
        x0 = np.random.default_rng(2).laplace(size=n) * 1e-3
        t = time.perf_counter()
        # config 4 costs ~1.7 ms per iteration: a fifth of the cap keeps the run within a minute
        _, info = m.map_estimate(x0, tol=1e-8, maxiter=args.maxiter // 5 if c == 4 else args.maxiter)
        r["to_tol_1e-8"] = {"iterations": info["iterations"], "converged": info["converged"],
                            "wall_s": time.perf_counter() - t, "F": info["F"],
                            "last_relative_change": float(info["relative_change"][-1].max())}
        del m
        torch.cuda.empty_cache()
        try:
            m64, _ = make(c, 64)
            r["fista_ms_per_iteration_64_chains"] = fista_ms(m64, 100 if c in (1, 3) else 50)
            del m64
        except torch.OutOfMemoryError as e:
            r["fista_ms_per_iteration_64_chains"] = f"not measured: {str(e).splitlines()[0]}"
        torch.cuda.empty_cache()
        res[f"config{c}"] = r
        print(json.dumps({f"config{c}": r}), flush=True)
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
