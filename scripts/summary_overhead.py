"""Cost of the streaming posterior summaries on one GPU (DESIGN.md 5 and 7b).

1. `k_stats_accumulate` at the bench shape (64 chains x 398 342 coefficients, L = 256, B = 1.5) in its three modes:
   CUDA events over `--launches` launches on accumulators larger than L2 (1.6-3.3 GB), bytes from the shapes, and the
   rate against a device-to-device copy of the same number of bytes timed in the same process.
2. The bench workload's `run()` (64 chains, L = 256, B = 1.5, Philox noise, Gram form, nsamples = 200,
   track = ["logposterior"]) at ngap 1 and 10, with and without summarise=("chain",), alternated `--reps` times: the
   time per iteration of the loop, and apart from it the one-off summary at the end of run().

usage: python scripts/summary_overhead.py <outdir> [--launches 200] [--reps 5]
Prints the card's name and power limit beside the numbers and writes <outdir>/summary_overhead.json.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else ""}


def accumulate_bytes(n, nch, mode):
    """bytes one push moves (every sample inside a batch, not at its first or last sample): the complex sample, then
    per slot the half-chain mean and M2 read and written and the open batch sum read and written"""
    slots = 1 if mode == 0 else 2
    return nch * n * (16 + slots * (32 + 16))


def time_kernel(n, nch, launches):
    import torch

    from pxmcmc_b200 import device as D

    out = {}
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.complex(torch.randn((nch, n), generator=g, device="cuda", dtype=torch.float64),
                      torch.randn((nch, n), generator=g, device="cuda", dtype=torch.float64))
    nsamples = 10_000  # b = 100: the timed pushes j = 1 .. 98 + k 100 fall inside batches (no fold, no first sample)
    for mode in (0, 1, 2):
        acc = D.stats_accumulator(n, nch, mode)
        js = [j for j in range(nsamples) if j % 100 not in (0, 99)][:launches]
        for j in js[:5]:
            D.stats_accumulate_dev(acc, x, mode, nsamples, j=j)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for j in js:
            D.stats_accumulate_dev(acc, x, mode, nsamples, j=j)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / len(js)
        nbytes = accumulate_bytes(n, nch, mode)
        # a copy of the same number of bytes (read + write), same process
        half = nbytes // 2 // 8
        src = torch.empty(half, dtype=torch.float64, device="cuda").fill_(1.0)
        dst = torch.empty_like(src)
        for _ in range(3):
            dst.copy_(src)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(len(js)):
            dst.copy_(src)
        c1.record()
        c1.synchronize()
        cms = c0.elapsed_time(c1) / len(js)
        out[f"mode{mode}"] = {"accumulator_bytes": acc.numel() * 8, "bytes_per_push": nbytes, "ms_per_push": ms,
                              "GBps": nbytes / ms / 1e6, "copy_ms": cms, "copy_GBps": 2 * half * 8 / cms / 1e6,
                              "fraction_of_copy": (nbytes / ms) / (2 * half * 8 / cms), "launches": len(js)}
        print(f"k_stats_accumulate mode {mode}: {ms:.4f} ms/push, {nbytes / ms / 1e6:.0f} GB/s; same-size copy "
              f"{2 * half * 8 / cms / 1e6:.0f} GB/s -> {out[f'mode{mode}']['fraction_of_copy']:.3f} of the copy", flush=True)
        del acc, src, dst
        torch.cuda.empty_cache()
    return out


def time_runs(L, B, J, nch, nsamples, reps):
    import torch

    from pxmcmc_b200 import sht
    from pxmcmc_b200.forward import SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1

    rng = np.random.default_rng(0)
    flm = rng.standard_normal(L * L) + 1j * rng.standard_normal(L * L)
    data = sht.inverse(flm, L).ravel()
    data = data / np.sqrt(np.mean(np.abs(data) ** 2))
    op = SphericalWaveletTransformOperator(data, 1.0, "synthesis", L, B, J, nchains=nch)
    assert op._ring_kind() == "harm"
    start = rng.laplace(size=(nch, op.nparams)) * 0.01
    res = {}
    for ngap in (1, 10):
        iters = (nsamples - 1) * ngap + 1
        times, finals = {"none": [], "chain": []}, []
        for rep in range(reps + 1):  # rep 0: warm-up (tables, graph pools)
            for key in ("none", "chain"):
                prm = PxMCMCParams(nsamples=nsamples, nburn=0, ngap=ngap, delta=1e-6, lmda=1e-6, mu=1.0, verbosity=0,
                                   track=["logposterior"])
                reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 1e-6, L=L, B=B, J_min=J)
                m = MYULA(op, reg, prm, noise="device", nchains=nch, seed=1234,
                          summarise=None if key == "none" else ("chain",))
                fin = [0.0]
                if key == "chain":  # the end-of-run reduction (partials, per-chain arrays to the host) timed apart
                    end = m._stats_end

                    def timed_end(end=end, fin=fin):
                        torch.cuda.synchronize()
                        t = time.perf_counter()
                        end()
                        torch.cuda.synchronize()
                        fin[0] = time.perf_counter() - t

                    m._stats_end = timed_end
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                m.run(start)
                torch.cuda.synchronize()
                dt = (time.perf_counter() - t0 - fin[0]) * 1e3 / iters
                if rep:
                    times[key].append(dt)
                    if key == "chain":
                        finals.append(fin[0] * 1e3)
                del m
        med = {k: float(np.median(v)) for k, v in times.items()}
        res[f"ngap{ngap}"] = {"iterations": iters, "ms_per_iteration": times, "median": med,
                              "overhead": med["chain"] / med["none"] - 1, "summary_at_end_ms": finals}
        print(f"run() ngap={ngap}: {med['none']:.4f} ms/iteration without, {med['chain']:.4f} with summarise=('chain',) "
              f"-> {100 * res[f'ngap{ngap}']['overhead']:+.2f} %  (all: {times}); summary at the end of run(): "
              f"{np.median(finals):.0f} ms (partials, per-chain arrays to the host, finalize)", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--nsamples", type=int, default=200)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("summary_overhead.py measures on a CUDA device; none is visible")
    os.makedirs(a.outdir, exist_ok=True)
    info = card()
    print(f"card: {info}", flush=True)
    from pxmcmc_b200 import device as D

    D.dev()
    out = {"card": info, "shape": {"L": 256, "B": 1.5, "nchains": 64, "n": 398342}}
    out["kernel"] = time_kernel(398342, 64, a.launches)
    out["run"] = time_runs(256, 1.5, 2, 64, a.nsamples, a.reps)
    with open(os.path.join(a.outdir, "summary_overhead.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
