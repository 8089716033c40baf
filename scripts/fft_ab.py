"""A/B of the persistent ring-FFT kernels for Bluestein lengths 512 / 1024 on the bench workload, in one process:
the two-CTA kernel `pxm_ring_fft3_kernel` (debug FFT mode 4) against the default one-CTA-per-SM `pxm_ring_fft6_kernel`.

Same setup as bench.py's measure_chains: 64 MYULA chains at L = 256, B = 1.5, J_min = 2, device noise, predictions
carried as ring coefficients.  Rounds alternate the two kernels; every round starts from the same chain state and
Philox step and measures
  (a) the ring-FFT stage per step from the library profiler (pxm_profile_begin / _end, kind 1), over --prof-steps,
  (b) the full step from CUDA events around --steps iterations, profiler off.
Before timing, three iterations under each kernel are compared with np.array_equal (state and pixel predictions).
Prints the GPU name and power limit (read-only nvidia-smi query), then medians and spreads; --json writes them too.

usage: python scripts/fft_ab.py [--rounds 5] [--steps 200] [--prof-steps 50] [--json out.json]
(PXM_LIB=<path> selects another build of the library)
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

KERNELS = {"two_cta_fft3": 4, "one_cta_fft6": 0}  # name -> pxm_debug_set_fft_multipass mode


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--prof-steps", type=int, default=50)
    ap.add_argument("--chains", type=int, default=64)
    ap.add_argument("--json")
    args = ap.parse_args()

    import torch

    import bench
    from pxmcmc_b200 import _lib, device as D, sht
    from pxmcmc_b200.forward import SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1

    torch.cuda.set_device(0)
    L, B, J, nch = 256, 1.5, 2, args.chains
    data = sht.inverse(bench.synthetic_flm(L), L).ravel()
    data = data / np.sqrt(np.mean(np.abs(data) ** 2))
    op = SphericalWaveletTransformOperator(data, 1.0, "synthesis", L, B, J, nchains=nch)
    prm = PxMCMCParams(nsamples=1, nburn=0, ngap=1, delta=1e-6, lmda=1e-6, mu=1.0, verbosity=0, track=[])
    reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, prm.lmda * prm.mu, L=L, B=B, J_min=J)
    m = MYULA(op, reg, prm, noise="device", nchains=nch, seed=1234, stream0=0).engine
    m.forward.fuse_ring = True
    X0 = D.to_dev_c(np.random.default_rng(7).laplace(size=(nch, m.forward.nparams)))
    P0 = m._initial_preds(X0)
    assert m._ring_mode()
    step0 = m._step_counter

    def set_kernel(name):
        _lib.check(_lib.lib.pxm_debug_set_fft_multipass(KERNELS[name]))

    def iterate(n):
        X, P = X0.clone(), P0.clone()
        m._step_counter = step0
        for _ in range(n):
            X, P = m.iterate(X, P)
        return X, P

    # ---- outputs: old vs new, bit for bit
    outs = {}
    for name in KERNELS:
        set_kernel(name)
        X, P = iterate(3)
        torch.cuda.synchronize()
        outs[name] = (D.to_host(X), D.to_host(m._pix(P)))
    a, b = outs.values()
    same = bool(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]))
    print(f"GPU: {gpu_identity()}")
    print(f"outputs after 3 iterations, {nch} chains: state and predictions bit-identical: {same}", flush=True)

    # ---- warm-up: every kernel for >= 0.3 s (clocks leave idle, modules loaded)
    for name in KERNELS:
        set_kernel(name)
        t = time.perf_counter()
        while time.perf_counter() - t < 0.3:
            iterate(5)
            torch.cuda.synchronize()

    res = {name: {"step_ms": [], "ring_fft_ms": []} for name in KERNELS}
    for r in range(args.rounds):
        for name in KERNELS:
            set_kernel(name)
            iterate(3)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            X, P = X0.clone(), P0.clone()
            m._step_counter = step0
            e0.record()
            for _ in range(args.steps):
                X, P = m.iterate(X, P)
            e1.record()
            torch.cuda.synchronize()
            res[name]["step_ms"].append(e0.elapsed_time(e1) / args.steps)
            _lib.check(_lib.lib.pxm_profile_begin(16 * args.prof_steps + 64))
            X, P = X0.clone(), P0.clone()
            m._step_counter = step0
            for _ in range(args.prof_steps):
                X, P = m.iterate(X, P)
            ms = (C.c_double * 3)()
            cnt = (C.c_longlong * 3)()
            _lib.check(_lib.lib.pxm_profile_end(ms, cnt))
            res[name]["ring_fft_ms"].append(ms[1] / args.prof_steps)
            print(f"round {r} {name}: step {res[name]['step_ms'][-1]:.4f} ms, ring FFT {res[name]['ring_fft_ms'][-1]:.4f} ms "
                  f"({cnt[1] // args.prof_steps} launches per step)", flush=True)
    _lib.check(_lib.lib.pxm_debug_set_fft_multipass(0))

    summary = {"gpu": gpu_identity(), "chains": nch, "steps": args.steps, "prof_steps": args.prof_steps, "rounds": args.rounds,
               "bit_identical": same}
    for name, v in res.items():
        for k, xs in v.items():
            summary[f"{name}.{k}"] = {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)),
                                      "all": [round(x, 5) for x in xs]}
    o, n = summary["two_cta_fft3.step_ms"]["median"], summary["one_cta_fft6.step_ms"]["median"]
    of, nf = summary["two_cta_fft3.ring_fft_ms"]["median"], summary["one_cta_fft6.ring_fft_ms"]["median"]
    summary["step_speedup"] = o / n
    summary["ring_fft_ratio"] = nf / of
    for name in KERNELS:
        s, f = summary[f"{name}.step_ms"], summary[f"{name}.ring_fft_ms"]
        print(f"{name}: step median {s['median']:.4f} ms [{s['min']:.4f}, {s['max']:.4f}]   "
              f"ring FFT median {f['median']:.4f} ms [{f['min']:.4f}, {f['max']:.4f}]")
    print(f"step time old / new = {o / n:.4f}; ring FFT new / old = {nf / of:.4f}")
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(summary, fh, indent=1)
    if not same:
        sys.exit("outputs differ between the kernels")


if __name__ == "__main__":
    main()
