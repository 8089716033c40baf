"""Rate of the rank-normalised diagnostics (pxm_rank_diagnostics) on AR(1) phi = 0.9 columns.

For every (m, n) shape, with --ncols columns (default 65 536, so that every input is larger than the 126 MB L2):
  kernel_ms   CUDA events around pxm_rank_diagnostics (transposition + per-column kernel) on a device-resident input,
              median of --reps calls after one warm-up call;
  e2e_ms      diagnostics.rank_diagnostics on the same samples as a host numpy array (uploads in 2 GB blocks included);
  oracle_ms_per_col  oracle/rank_diagnostics_ref.py on --check columns, one host core.
Before timing, the device outputs of --check seeded columns are compared with the oracle (R-hat 1e-12 absolute, ESS
1e-10 relative).  DRAM bytes: the transposition reads and writes the block once, the per-column kernel reads its column
once from DRAM (its three reloads of the 128 KB column hit L2), so at least 3 x 8 S bytes per column.
Prints one JSON line, with the card's name and power limit read in the same run.

    python scripts/rank_diagnostics_rate.py [--ncols 65536] [--reps 5] [--check 64] [--out FILE]
"""
import os

os.environ.setdefault("OMP_NUM_THREADS", "1")
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
os.environ.setdefault("MKL_NUM_THREADS", "1")

import argparse  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # the torch name is still recorded below
        return None, f"unavailable ({e})"


def ar1_dev(torch, m, n, ncols, phi, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.empty((m, n, ncols), dtype=torch.float64, device="cuda")
    x[:, 0] = torch.randn((m, ncols), generator=g, dtype=torch.float64, device="cuda") / (1 - phi ** 2) ** 0.5
    for t in range(1, n):
        x[:, t] = phi * x[:, t - 1] + torch.randn((m, ncols), generator=g, dtype=torch.float64, device="cuda")
    return x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncols", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--check", type=int, default=64)
    ap.add_argument("--shapes", default="4x1000,64x256,8x2048")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from oracle import rank_diagnostics_ref as K
    from pxmcmc_b200 import device as D
    from pxmcmc_b200 import diagnostics
    from pxmcmc_b200._lib import check, lib, ptr, stream_ptr

    if not torch.cuda.is_available():
        raise SystemExit("rank_diagnostics_rate: needs a CUDA device")
    D.dev()
    name, limit = card()
    res = {"metric": "rank_diagnostics_rate", "gpu": name or torch.cuda.get_device_name(), "power_limit": limit,
           "phi": 0.9, "ncols": a.ncols, "shapes": []}
    for k, shape in enumerate(a.shapes.split(",")):
        m, n = (int(v) for v in shape.split("x"))
        S = m * n
        x = ar1_dev(torch, m, n, a.ncols, 0.9, seed=100 + k)
        x2 = x.view(S, a.ncols)
        scratch = torch.empty(lib.pxm_rank_diagnostics_scratch_doubles(m, n, a.ncols), dtype=torch.float64,
                              device=x.device)
        out = torch.full((3, a.ncols), -7.0, dtype=torch.float64, device=x.device)

        def call():
            check(lib.pxm_rank_diagnostics(ptr(x2), m, n, a.ncols, a.ncols, ptr(scratch), ptr(out[0]), ptr(out[1]),
                                           ptr(out[2]), stream_ptr()))

        call()
        torch.cuda.synchronize()
        cols = np.sort(np.random.default_rng(k).choice(a.ncols, a.check, replace=False))
        xs = x[:, :, torch.from_numpy(cols).to(x.device)].cpu().numpy()
        got = out[:, torch.from_numpy(cols).to(x.device)].cpu().numpy()
        t0 = time.perf_counter()
        ref = np.array(K.rank_diagnostics(xs))
        oracle_ms = (time.perf_counter() - t0) * 1e3 / a.check
        d_rhat = float(np.max(np.abs(got[0] - ref[0])))
        d_ess = float(np.max(np.abs(got[1:] - ref[1:]) / np.abs(ref[1:])))
        if not (d_rhat <= 1e-12 and d_ess <= 1e-10):
            raise SystemExit(f"rank_diagnostics_rate: {shape}: device differs from the oracle (R-hat {d_rhat:.2e}, "
                             f"ESS {d_ess:.2e})")
        times = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        kernel_ms = float(np.median(times))
        host = x.cpu().numpy()
        del scratch
        t0 = time.perf_counter()
        e2e = diagnostics.rank_diagnostics(host)
        e2e_ms = (time.perf_counter() - t0) * 1e3
        assert np.array_equal(e2e.ess_bulk, out[1].cpu().numpy())
        dram = 3 * 8 * S * a.ncols
        res["shapes"].append({
            "m": m, "n": n, "input_bytes": 8 * S * a.ncols, "kernel_ms": round(kernel_ms, 3),
            "kernel_ms_all": [round(t, 3) for t in times], "e2e_ms": round(e2e_ms, 1),
            "us_per_col": round(kernel_ms * 1e3 / a.ncols, 4), "min_dram_bytes": dram,
            "min_dram_GBps": round(dram / kernel_ms / 1e6, 1), "oracle_ms_per_col": round(oracle_ms, 3),
            "speedup_kernel_vs_oracle_core": round(oracle_ms * a.ncols / kernel_ms, 1),
            "speedup_e2e_vs_oracle_core": round(oracle_ms * a.ncols / e2e_ms, 1),
            "check_cols": a.check, "max_abs_d_rhat": d_rhat, "max_rel_d_ess": d_ess,
            "median_ess_bulk_over_theory": round(float(np.median(got[1])) / (S * 0.1 / 1.9), 3)})
        del x, x2, out, host
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
