"""Regenerate profiles/traffic_r2.json: DRAM traffic per launch of the dominant kernels, measured with ncu
(dram__bytes_read.sum + dram__bytes_write.sum) on the bench workloads, keyed to the hash of the kernel sources
(bench.py reports `traffic` from this file and says whether the sources have changed since).

Run on the GPU box AFTER the same commands have exited 0 without ncu:
    gpurun -- 'python bench.py --no-extras --no-cpu-baseline && python scripts/refresh_traffic.py'
writes gpurun_out/traffic_r2.json (copy it to profiles/) and gpurun_out/traffic_r2_launches.csv."""
import csv
import io
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

METRICS = "dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum"


def ncu(cmd, kernel_regex, skip, count):
    full = ["ncu", "--metrics", METRICS, "--clock-control", "none", "-k", f"regex:{kernel_regex}", "--launch-skip", str(skip),
            "--launch-count", str(count), "--csv"] + cmd
    r = subprocess.run(full, capture_output=True, text=True, cwd=ROOT)
    rows = [row for row in csv.reader(io.StringIO(r.stdout)) if len(row) > 14 and row[0].isdigit()]
    out = {}
    for row in rows:
        d = out.setdefault(int(row[0]), {"kernel": row[4].split("(")[0]})
        val = float(row[14].replace(",", ""))
        unit = row[13].lower()
        if "byte" in unit:
            val *= {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1)
        d[row[12]] = val
    return [out[k] for k in sorted(out)], r.stdout


def main():
    py = sys.executable
    chains = [py, "bench.py", "--steps", "3", "--warmup", "3", "--no-extras", "--no-cpu-baseline", "--blocks", "0", "--e2e-steps", "1"]
    wl = [py, "bench.py", "--workload", "wl-msharded", "--steps", "3", "--warmup", "3"]
    res = {"csrc_sha": bench.csrc_sha(), "how": "ncu --metrics " + METRICS + " --clock-control none; bytes = dram read + write per launch"}
    logs = []
    # one full MYULA step = 4 ring-FFT launches of the persistent kernel and 4 Legendre launches; skip the plan set-up and
    # the first steps (the Legendre kernel also builds the quadrature tables at plan creation: skip generously)
    # (the bench carries the predictions in harmonic form: 2 persistent ring-FFT launches and 3 Legendre launches per step;
    # two consecutive steps are captured)
    fft, log = ncu(chains, "pxm_ring_fft6_kernel", 12, 4)
    logs.append(log)
    leg, log = ncu(chains, "pxm_legendre_kernel", 60, 6)
    logs.append(log)
    wleg, log = ncu(wl, "pxm_legendre_kernel", 400, 4)
    logs.append(log)

    def total(d):
        return d.get("dram__bytes_read.sum", 0.0) + d.get("dram__bytes_write.sum", 0.0)

    if fft:
        res["ring_fft_bytes_per_stage"] = sum(total(d) for d in fft) / len(fft)
        res["ring_fft_launches"] = [{"bytes": total(d), "us": d.get("gpu__time_duration.sum", 0) / 1e3} for d in fft]
    if leg:
        res["legendre_bytes_per_launch"] = sum(total(d) for d in leg) / len(leg)
        res["legendre_launches"] = [{"bytes": total(d), "us": d.get("gpu__time_duration.sum", 0) / 1e3} for d in leg]
    if wleg:
        res["wl_legendre_bytes_per_iteration"] = sum(total(d) for d in wleg)
        res["wl_legendre_launches"] = [{"bytes": total(d), "us": d.get("gpu__time_duration.sum", 0) / 1e3} for d in wleg]
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(res, open(os.path.join(ROOT, "gpurun_out", "traffic_r2.json"), "w"), indent=1)
    open(os.path.join(ROOT, "gpurun_out", "traffic_r2_launches.csv"), "w").write("\n".join(logs))
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
