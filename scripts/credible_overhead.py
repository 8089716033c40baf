"""Cost of the streaming credible intervals on one GPU (DESIGN.md 5 and 7b).

1. `k_credible_push` at the bench shape (64 chains x 398 342 coefficients, L = 256, B = 1.5) in its three modes, at
   N = 64 x 200 and 64 x 1 000 pooled samples (mode 2: 128 logical chains, twice that), alpha = 0.05: CUDA events
   around every push of a complete run of pushes on fresh iid normal samples, reported separately for the fill phase
   (pooled count < K) and the steady state.  The heaps (2.1-20 GB) are far larger than L2.  The same pushes are timed
   with the [slot][column] heap layout (a variant library built with -DPXM_CREDIBLE_SLOT_MAJOR in a temporary
   directory, run in a child process).
2. The bench workload's `run()` (64 chains, L = 256, B = 1.5, Philox noise, Gram form, nsamples = 200,
   track = ["logposterior"]) at ngap 1 and 10, with and without credible=("chain",), alternated `--reps` times: the
   time per iteration of the loop, and apart from it
3. the finalize at the end of run() (one pxm_credible_finalize, intervals to the host).

usage: python scripts/credible_overhead.py <outdir> [--reps 3] [--no-variant]
Prints the card's name and power limit beside the numbers and writes <outdir>/credible_overhead.json.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
N_COEF, NCH = 398342, 64


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else ""}


def time_pushes(alpha=0.05):
    import torch

    from pxmcmc_b200 import device as D
    from pxmcmc_b200.diagnostics import credible_tails

    out = {}
    g = torch.Generator(device="cuda").manual_seed(0)
    for nsamples in (200, 1000):
        for mode in (0, 1, 2):
            parts = 2 if mode == 2 else 1
            tails = credible_tails(NCH * parts * nsamples, alpha)
            N, lo_a, _, lo_b, _ = tails
            klo = min(lo_a + 2, N)
            st = D.credible_state(N_COEF, mode, tails)
            x = torch.empty((NCH, N_COEF), dtype=torch.complex128, device="cuda")
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nsamples)]
            fill = []
            for j in range(nsamples):
                torch.view_as_real(x).normal_(generator=g)
                fill.append(j * NCH * parts < klo)
                ev[j][0].record()
                D.credible_push_dev(st, x, mode, tails, j * NCH * parts)
                ev[j][1].record()
            torch.cuda.synchronize()
            ms = np.array([a.elapsed_time(b) for a, b in ev])
            fill = np.array(fill)
            t0 = time.perf_counter()
            D.credible_finalize_dev(st, N_COEF, mode, tails)
            torch.cuda.synchronize()
            fin = (time.perf_counter() - t0) * 1e3
            r = {"npooled": N, "K_per_tail": klo, "heap_bytes": st.numel() * 8, "state_bytes_read": NCH * N_COEF * 16,
                 "fill_pushes": int(fill.sum()), "fill_ms_per_push": float(ms[fill].mean()),
                 "steady_ms_per_push": float(ms[~fill].mean()), "steady_first10_ms": float(ms[~fill][:10].mean()),
                 "steady_last10_ms": float(ms[~fill][-10:].mean()), "total_push_ms": float(ms.sum()),
                 "finalize_ms_host_clock": fin}
            out[f"n{nsamples}_mode{mode}"] = r
            print(f"  k_credible_push mode {mode} N = {N} (K = {klo}, heaps {r['heap_bytes'] / 1e9:.2f} GB): fill "
                  f"{r['fill_ms_per_push']:.3f} ms/push ({r['fill_pushes']} pushes), steady {r['steady_ms_per_push']:.3f} "
                  f"ms/push (first 10 {r['steady_first10_ms']:.3f}, last 10 {r['steady_last10_ms']:.3f}); "
                  f"state read at {r['state_bytes_read'] / r['steady_last10_ms'] / 1e6:.0f} GB/s late in the run; "
                  f"finalize {fin:.2f} ms", flush=True)
            del st, x
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
                          credible=None if key == "none" else ("chain",))
                fin = [0.0]
                if key == "chain":  # the end-of-run finalize (intervals to the host) timed apart
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
                torch.cuda.empty_cache()
        med = {k: float(np.median(v)) for k, v in times.items()}
        res[f"ngap{ngap}"] = {"iterations": iters, "ms_per_iteration": times, "median": med,
                              "overhead": med["chain"] / med["none"] - 1, "finalize_at_end_ms": finals}
        print(f"run() ngap={ngap}: {med['none']:.4f} ms/iteration without, {med['chain']:.4f} with credible=('chain',) "
              f"-> {100 * res[f'ngap{ngap}']['overhead']:+.2f} %  (all: {times}); finalize at the end of run(): "
              f"{np.median(finals):.1f} ms", flush=True)
    return res


def variant_pushes():
    """the pushes of time_pushes() with the [slot][column] heap layout, in a child process on a variant library"""
    with tempfile.TemporaryDirectory() as tmp:
        so = os.path.join(tmp, "libpxmcmc_b200_slot_major.so")
        subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "build_variant.py"), so,
                        "-DPXM_CREDIBLE_SLOT_MAJOR", "pxm_credible.cu"], check=True, capture_output=True)
        js = os.path.join(tmp, "pushes.json")
        subprocess.run([sys.executable, os.path.abspath(__file__), tmp, "--pushes-only", js], check=True,
                       env=dict(os.environ, PXM_LIB=so))
        with open(js) as f:
            return json.load(f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--nsamples", type=int, default=200)
    ap.add_argument("--no-variant", action="store_true")
    ap.add_argument("--pushes-only", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("credible_overhead.py measures on a CUDA device; none is visible")
    from pxmcmc_b200 import device as D

    D.dev()
    if a.pushes_only:
        print("[slot][column] heap layout:", flush=True)
        with open(a.pushes_only, "w") as f:
            json.dump(time_pushes(), f)
        return
    os.makedirs(a.outdir, exist_ok=True)
    info = card()
    print(f"card: {info}", flush=True)
    out = {"card": info, "shape": {"L": 256, "B": 1.5, "nchains": NCH, "n": N_COEF}, "alpha": 0.05}
    print("[column][slot] heap layout (the library's):", flush=True)
    out["push_column_major"] = time_pushes()
    if not a.no_variant:
        out["push_slot_major"] = variant_pushes()
    out["run"] = time_runs(256, 1.5, 2, NCH, a.nsamples, a.reps)
    with open(os.path.join(a.outdir, "credible_overhead.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
