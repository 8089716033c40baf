"""Device time of one SKROCK stage, fused (`pxm_skrock_shift` / `pxm_skrock_stage`) against the composition it replaced
(`pxm_philox_normal` + `pxm_lincomb` + `pxm_gradlogpi` + `pxm_lincomb` at stage 1, `pxm_gradlogpi` + `pxm_lincomb` at
later stages), at 64 chains x 398 342 coefficients (L = 256 wavelet coefficients of the bench shape; every array larger
than L2) and at the config-3 single chain (76 068), and the per-step time of both schemes at config 3 (one CUDA graph
per step).  Prints one JSON object with the card's name and power limit; `--out FILE` also writes it there.

    python scripts/skrock_stage_timing.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def events_ms(fn, n, warm=10):
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


def stage_times(D, nch, n, reps):
    g = torch.Generator(device="cuda").manual_seed(1)

    def cn():
        return torch.complex(torch.randn(nch, n, dtype=torch.float64, device="cuda", generator=g),
                             torch.randn(nch, n, dtype=torch.float64, device="cuda", generator=g))

    U, V, gradg = cn(), cn(), cn()
    Tv = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    out = torch.empty_like(U)
    lmda, a, b, c, c0, cs, e = 5e-7, 1e-7, 1.9, -0.9, 0.0, 1e-3, 2e-3
    Z = D.SkrockNoise(seed=5, step=1)

    def fused_j():
        D.skrock_stage_dev(U, V, gradg, None, Tv, 0.0, lmda, a, b, c, c0, out=out)

    def composed_j():
        D.lincomb_dev([(a, D.gradlogpi_dev(U, None, Tv, 0.0, gradg, lmda)), (b, U), (c, V)], c0=c0, out=out)

    def fused_1():
        D.skrock_shift_dev(U, cs, Z, out=V)
        D.skrock_stage_dev(U, None, gradg, None, Tv, 0.0, lmda, a, 1.0, 0.0, 0.0, Z=Z, c_shift=cs, e=e, out=out)

    def composed_1():
        z = D.philox_normal_dev(nch, n, 5, 1)
        Y = D.lincomb_dev([(1.0, U)], z=z, cz=cs)
        D.lincomb_dev([(1.0, U), (a, D.gradlogpi_dev(Y, None, Tv, 0.0, gradg, lmda))], z=z, cz=e, out=out)

    # same-inputs check at this size: the reference-scheme stage is bit-identical
    fused_j()
    f = out.clone()
    composed_j()
    same_j = bool(torch.equal(f, out))
    fused_1()
    f = out.clone()
    composed_1()
    same_1 = bool(torch.equal(f, out))
    res = {"nchains": nch, "n": n, "bit_identical": {"stage_j": same_j, "stage_1": same_1}}
    for rnd in range(2):  # alternate the two versions
        for name, fn in (("fused_stage_j", fused_j), ("composed_stage_j", composed_j), ("fused_stage_1", fused_1),
                         ("composed_stage_1", composed_1)):
            res.setdefault(name + "_ms", []).append(events_ms(fn, reps))
    res = {k: (min(v) if k.endswith("_ms") else v) for k, v in res.items()}
    el = nch * n
    res["bytes_per_coefficient_model"] = {"fused_stage_j": 72, "composed_stage_j": 120, "fused_stage_1": 88,
                                          "composed_stage_1": 160}
    for k in ("fused_stage_j", "composed_stage_j", "fused_stage_1", "composed_stage_1"):
        res[k + "_model_TBps"] = res["bytes_per_coefficient_model"][k] * el / (res[k + "_ms"] * 1e-3) / 1e12
    del U, V, gradg, out
    torch.cuda.empty_cache()
    return res


def config3_steps(reps):
    from pxmcmc_b200 import device as D
    from pxmcmc_b200 import paths
    from pxmcmc_b200.forward import PathIntegralOperator
    from pxmcmc_b200.mcmc import SKROCK, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1_Power_Weights

    L, B, s = 128, 2, 10
    rng = np.random.default_rng(7)
    z = rng.uniform(-1, 1, size=(10000, 2))
    lon = rng.uniform(-180, 180, size=(10000, 2))
    lat = np.degrees(np.arcsin(z))
    A = paths.get_path_matrix(np.stack([lat[:, 0], lon[:, 0]], 1), np.stack([lat[:, 1], lon[:, 1]], 1), L)
    y = A @ rng.standard_normal(A.shape[1]) + 0.05 * rng.standard_normal(A.shape[0])
    op = PathIntegralOperator(A, y, np.full(A.shape[0], 0.05), "synthesis", L, B, 2)
    prm = PxMCMCParams(delta=1e-6, lmda=5e-7, mu=1.0, s=s, verbosity=0, nsamples=1, track=[])
    reg = S2_Wavelets_L1_Power_Weights("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-7, L=L, B=B,
                                       J_min=2, eta=1)
    graphs = {sch: SKROCK(op, reg, prm, scheme=sch, noise="device", seed=5).capture(D.to_dev_c(np.zeros((1, op.nparams))))
              for sch in ("reference", "published")}
    out = {}
    for _ in range(3):
        for sch, g in graphs.items():
            out.setdefault(sch + "_ms_per_step", []).append(events_ms(g.step, reps))
    return {k: min(v) for k, v in out.items()} | {"nparams": op.nparams, "nnz": int(A.nnz), "s": s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from pxmcmc_b200 import device as D

    res = {"card": card(), "method": "CUDA events around `reps` back-to-back launches, best of alternated rounds"}
    res["stage_64x398342"] = stage_times(D, 64, 398342, args.reps)
    res["stage_config3_single_chain"] = stage_times(D, 1, 76068, args.reps * 10)
    res["config3_step"] = config3_steps(args.reps)
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
