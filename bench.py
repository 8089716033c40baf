#!/usr/bin/env python
"""Benchmark of the proximal-Langevin hot path (BASELINE.json metric:
"MYULA iterations/s at L=256 (per chain and x chains)").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one MYULA iteration (mcmc.py:158-164 of the reference: data-fidelity
gradient through Psi^dagger, fused soft-threshold prox + Langevin update with
Philox noise, new predictions through Psi) of `--chains` independent chains per
GPU, wavelet-synthesis operator at L=256, B=1.5, J_min=2 (398 342 complex
coefficients and 130 816 complex pixels per chain), synthetic complex map.
Chains are independent units: weak scaling, no data-path collective.

Prints ONE JSON line (see DESIGN.md "Measurement" for every field).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L_DEF, B_DEF, JMIN_DEF = 256, 1.5, 2
METRIC = "MYULA chain-iterations/s at L=256 (x chains)"
UNIT = "chain-iterations/s"


def bandlimits(L, B, J_min):
    J = int(np.ceil(np.log(L) / np.log(B)))
    out = [min(int(np.ceil(B ** J_min)), L)]
    for j in range(J_min, J + 1):
        out.append(min(int(np.ceil(B ** (j + 1))), L))
    return out


def workload_name(L, B, J_min):
    """the same string in both arms (ours and --impl reference): the driver compares the configurations"""
    return (f"MYULA L={L} B={B} J_min={J_min} synthesis, Identity measurement, S2_Wavelets_L1 "
            "(config 5 of BASELINE.json: independent chains, chain-iterations/s)")


def algorithmic_flops_per_chain_iteration(L, B, J_min):
    """SURVEY.md 8(d): F_it = 2 F_Psi = 8 (L^3 + sum_scales L_j^3) FP64 flops (FFT flops excluded)."""
    return 8.0 * (L ** 3 + sum(b ** 3 for b in bandlimits(L, B, J_min)))


def synthetic_flm(L, seed=20240):
    rng = np.random.default_rng(seed)
    flm = np.zeros(L * L, dtype=complex)
    for el in range(L):
        amp = (1.0 + el) ** -1.25  # C_l = (1+l)^-2.5
        flm[el * el + el] = amp * rng.standard_normal()
        m = np.arange(1, el + 1)
        a = amp * (rng.standard_normal(el) + 1j * rng.standard_normal(el)) / np.sqrt(2)
        flm[el * el + el + m] = a
        flm[el * el + el - m] = (-1.0) ** m * np.conj(a)
    return flm


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region"""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit())}


# ---------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the CPU oracle restatement of the reference path
# ---------------------------------------------------------------------------------------
def _oracle_one_iteration(args):
    L, B, J_min, seed = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=1)
    except Exception:  # noqa: BLE001
        ctx = None
    from oracle import pxmcmc_ref as R
    from oracle import ssht_ref

    rng = np.random.default_rng(seed)
    t = R.WaveletTransform(L, B, J_min)
    data = ssht_ref.inverse(synthetic_flm(L), L, 0).ravel()
    data = data / np.sqrt(np.mean(np.abs(data) ** 2))
    op = R.ForwardOperator(data, 1.0, "synthesis", t, R.IdentityMeasurement(data.size, data.size), t.ncoefs)
    prior = R.S2WaveletsL1("synthesis", t.inverse, t.inverse_adjoint, 1e-6, L, B, J_min)
    X = rng.laplace(size=t.ncoefs)
    preds = op.forward(X)
    reps = int(os.environ.get("PXM_ORACLE_REPS", "1"))
    t0 = time.perf_counter()
    for _ in range(reps):
        X, preds = R.myula_iteration(op, prior, 1e-6, 1e-6, X, preds, rng.standard_normal(t.ncoefs))[:2]
    dt = (time.perf_counter() - t0) / reps
    if ctx is not None:
        ctx.unregister() if hasattr(ctx, "unregister") else None
    return dt


def cpu_reference_throughput(L, B, J_min, procs, steps):
    """`steps` rounds of `procs` independent chain-iterations run one per host core"""
    import multiprocessing as mp

    times = []
    with mp.get_context("spawn").Pool(procs) as pool:
        for s in range(steps):
            t0 = time.perf_counter()
            pool.map(_oracle_one_iteration, [(L, B, J_min, 1000 * s + i) for i in range(procs)])
            times.append(time.perf_counter() - t0)
    # the timed map includes building each worker's inputs; use the workers' own timers instead
    return times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the CPU leg is O(L^3) numpy: bound the sample so that the run ends within minutes
    L = args.ref_L
    procs = max(1, min(os.cpu_count() or 1, args.ref_procs))
    import multiprocessing as mp

    steps = max(1, min(args.steps, 2))
    t_iter = []
    with mp.get_context("spawn").Pool(procs) as pool:
        for s in range(args.warmup and 1 or 0):
            pool.map(_oracle_one_iteration, [(L, args.B, args.J_min, i) for i in range(procs)])
        t0 = time.perf_counter()
        for s in range(steps):
            t_iter += pool.map(_oracle_one_iteration, [(L, args.B, args.J_min, 100 * s + i) for i in range(procs)])
        wall = time.perf_counter() - t0
    mean_it = float(np.mean(t_iter))
    value = procs / mean_it  # procs chains advance one iteration every mean_it seconds
    scale = (algorithmic_flops_per_chain_iteration(args.L, args.B, args.J_min) /
             algorithmic_flops_per_chain_iteration(L, args.B, args.J_min))
    sample = (f"{steps} x {procs} chain-iterations of the numpy oracle (CPU restatement of the reference path), one per core, "
              f"at L={L}" + ("" if L == args.L else f"; value scaled by the O(L^3) flop ratio {scale:.1f} to L={args.L}"))
    value_at_L = value / scale
    line = {
        "impl": "reference", "metric": METRIC, "value": value_at_L, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * mean_it * scale, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.L, args.B, args.J_min),
                   "implementation": "CPU: numpy port of the reference's Python layer over a restatement of ssht / s2let, one chain per process"},
        "cpu_baseline": {"value": value_at_L, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": value_at_L, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": wall,
    }
    emit(line)


# ---------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def bind_to_gpu_numa_node(local):
    """pin this rank's threads to the CPUs next to its GPU BEFORE any pinned host buffer is allocated (first touch):
    the end-to-end path moves ~1 GB per step and GPU over PCIe, and host memory on the far socket halves that"""
    try:
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        return sorted(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001  (restricted cpuset, no NVML: keep the inherited affinity)
        return None


def csrc_sha():
    """hash of the kernel sources: ncu-derived numbers quoted by the bench line say which sources they were measured on"""
    import hashlib

    h = hashlib.sha256()
    d = os.path.join(ROOT, "pxmcmc_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".h")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def fft_stage_traffic(traffic, ring_mode):
    """mean DRAM bytes per executed ring-FFT stage: all four stages of the literal step, or only the two coefficient-side
    stages (the large ones) when the predictions are carried as ring coefficients"""
    ls = [d["bytes"] for d in traffic.get("ring_fft_launches", [])]
    if not ls:
        return traffic.get("ring_fft_bytes_per_stage")
    if ring_mode:
        big = [b for b in ls if b > 0.5 * max(ls)]
        return sum(big) / len(big)
    return sum(ls) / len(ls)


def load_traffic():
    """DRAM traffic per launch of the dominant kernels from the tracked ncu summary profiles/traffic_r2.json
    (regenerated by scripts/refresh_traffic.py under ncu); `current` says whether the kernels have changed since"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic_r2.json")))
    except Exception:  # noqa: BLE001
        return {}, {"file": None, "current": False}
    return t, {"file": "profiles/traffic_r2.json", "csrc_sha": t.get("csrc_sha"), "current": t.get("csrc_sha") == csrc_sha()}


class Ctx:
    """rank bookkeeping + the collectives the measurement itself needs (barrier, max over ranks)"""

    def __init__(self):
        import torch

        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.cpus = bind_to_gpu_numa_node(self.local)
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist

            # stdout carries ONE JSON line: NCCL's own log (version banner, NCCL_DEBUG=INFO topology / comm lines) goes to
            # stderr instead of being switched off
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
                os.environ["NCCL_DEBUG"] = "WARN"  # NCCL honours NCCL_DEBUG_FILE only above the VERSION level
            # belt and braces: while the communicator comes up (NCCL prints its banner at the first collective) this
            # process's stdout IS stderr
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
            self.dist = dist

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def reduce(self, vals, op="max"):
        if self.dist is None:
            return [float(v) for v in vals]
        t = self.torch.tensor([float(v) for v in vals], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def release_plans():
    """drop the cached plans (Legendre tables) of a finished workload"""
    import gc

    import torch

    from pxmcmc_b200 import device as D

    D.WaveletPlan._cache.clear()
    D.ShtPlan._cache.clear()
    D._scratch.clear()
    gc.collect()
    torch.cuda.empty_cache()


DUMP_SAMPLES = 1 << 20  # complex values kept per dumped array: 16 MiB of float64, 32 MiB for the two arrays


def sample_outputs(t):
    """float64 [k, 2] (real, imaginary parts) of a complex device tensor: all its elements in row-major order when there
    are at most DUMP_SAMPLES, else DUMP_SAMPLES of them at sorted flat indices drawn without replacement from a generator
    seeded with 0, i.e. the same elements for the same shape in every run"""
    import torch

    flat = t.reshape(-1)
    if flat.numel() > DUMP_SAMPLES:
        idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_SAMPLES, replace=False))
        flat = flat[torch.as_tensor(idx, device=flat.device)]
    return torch.view_as_real(flat).cpu().numpy()


def measure_chains(ctx, args, nch, total_chains, steps, blocks=0, block_iters=100, e2e_steps=0, real=False, dump=False):
    """`steps` MYULA iterations of `nch` chains on this GPU (config 5 / the BASELINE metric): device-resident value, per-stage
    device times, optional sustained blocks and the end-to-end figure through host buffers.  Chain c of the job draws
    Philox stream c whatever the sharding.  `real`: REAL-valued data (the drivers' `_mw_` input route,
    experiments/earthtopography/main.py:83-85) and MYULA(real_pairs=True): the `nch` real chains travel as nch / 2
    complex device chains.  `dump`: out["outputs"] holds samples (`sample_outputs`) of the chain states and pixel
    predictions the last timed step returned."""
    import ctypes as C

    torch = ctx.torch
    from pxmcmc_b200 import _lib, device as D, sht
    from pxmcmc_b200.forward import SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1
    from pxmcmc_b200.sharding import philox_stream0

    L, B, J_min = args.L, args.B, args.J_min
    data = sht.inverse(synthetic_flm(L), L).ravel()
    data = data / np.sqrt(np.mean(np.abs(data) ** 2))  # complex, as on the reference's HEALPix path
    if real:
        data = np.ascontiguousarray(data.real)
        data = data / np.sqrt(np.mean(data ** 2))
    op = SphericalWaveletTransformOperator(data, 1.0, "synthesis", L, B, J_min, nchains=nch)
    prm = PxMCMCParams(nsamples=1, nburn=0, ngap=1, delta=1e-6, lmda=1e-6, mu=1.0, verbosity=0, track=[])
    reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, prm.lmda * prm.mu, L=L, B=B, J_min=J_min)
    outer = MYULA(op, reg, prm, noise="device", nchains=nch, seed=1234, stream0=philox_stream0(total_chains, ctx.world, ctx.rank),
                  real_pairs=real)
    m = outer.engine  # the sampler that iterates on the device representation (nch / 2 packed chains when `real`)
    nch_dev = m.nchains
    op = m.forward
    ncoef, npix = op.nparams, L * (2 * L - 1)
    rng = np.random.default_rng(7 + ctx.rank)
    X = D.to_dev_c(rng.laplace(size=(nch, ncoef)))
    if real:
        X = outer.pack(X)
    # the form MYULA.run carries the predictions in: ring-Fourier coefficients of the image when the operator allows it
    # (Identity measurement, inverse covariance constant along rings: the pixel-side ring-FFT pair of consecutive
    # iterations cancels, DESIGN.md 3), pixels otherwise (--no-ring-fusion)
    op.fuse_ring = not args.no_ring_fusion
    P = m._initial_preds(X)
    ring_mode = m._ring_mode()
    pred_kind = op._ring_kind() if ring_mode else None
    for _ in range(max(args.warmup, 3)):
        X, P = m.iterate(X, P)
    # the GPU leaves its idle clocks only after some tens of ms of load: keep iterating (untimed)
    # until 0.3 s have passed so that the timed region starts at the sustained clock.  The timed region then restarts
    # from the state and Philox step reached after the warm-up iterations, so that its inputs do not depend on how
    # many iterations fitted into the 0.3 s
    X0, P0, step0 = X.clone(), P.clone(), m._step_counter
    t_w = time.perf_counter()
    while time.perf_counter() - t_w < 0.3:
        X, P = m.iterate(X, P)
        torch.cuda.synchronize()
    X, P, m._step_counter = X0, P0, step0
    del X0, P0
    ctx.barrier()
    sampler = ClockSampler(ctx.local)
    sampler.start()
    l0 = _lib.lib.pxm_launch_count()
    _lib.check(_lib.lib.pxm_profile_begin(16 * steps + 64))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record()
    for _ in range(steps):
        X, P = m.iterate(X, P)
    e1.record()
    ctx.barrier()
    last = (X, P)  # what the last timed step returned (the iterations below allocate new tensors)
    ms = e0.elapsed_time(e1)
    ms_kind = (C.c_double * 3)()
    cnt_kind = (C.c_longlong * 3)()
    _lib.check(_lib.lib.pxm_profile_end(ms_kind, cnt_kind))
    launches = _lib.lib.pxm_launch_count() - l0
    ms, leg, fft, el = ctx.reduce([ms, ms_kind[0], ms_kind[1], ms_kind[2]])
    out = {"nch": nch, "nch_dev": nch_dev, "ncoef": ncoef, "npix": npix, "ms": ms, "steps": steps, "launches": int(launches),
           "ring_mode": ring_mode, "pred_kind": pred_kind,
           "stage_ms": {"legendre": leg / steps, "ring_fft": fft / steps, "elementwise": el / steps},
           "counts": [int(c) for c in cnt_kind], "table_bytes": int(op.transform._plan(nch_dev).table_bytes)}
    # sustained rate: `blocks` blocks of `block_iters` iterations, each timed on the device; median over blocks of the
    # max over ranks (SURVEY.md 8(d): >= 1000 iterations, median of 5)
    if blocks:
        per_block = []
        for _ in range(blocks):
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ctx.barrier()
            b0.record()
            for _ in range(block_iters):
                X, P = m.iterate(X, P)
            b1.record()
            ctx.barrier()
            per_block.append(ctx.reduce([b0.elapsed_time(b1)])[0] / block_iters)
        out["sustained_ms_per_step"] = float(np.median(per_block))
        out["sustained_blocks_ms_per_step"] = [round(v, 5) for v in per_block]
    sampler.stop_flag = True
    sampler.join(timeout=2)
    out["clocks"] = sampler.summary()
    out["finite"] = bool(torch.isfinite(torch.view_as_real(X)).all().item())
    # ---- end to end through pinned host buffers, rank-local -------------------------------------------------
    if e2e_steps:
        # state in, state out: the chain state travels host -> device -> host every step; the predictions the gradient
        # needs are recomputed from the state on the device (MYULA.iterate_host(X): as `chain_step` of the reference,
        # a state is mapped to a state).  `--e2e-with-preds` also moves the pixel-space predictions both ways (round 1's form).
        with_preds = bool(getattr(args, "e2e_with_preds", False))
        Xh = torch.empty((nch_dev, ncoef), dtype=torch.complex128).pin_memory()
        Xh.copy_(X.cpu())
        Xo = torch.empty_like(Xh).pin_memory()
        Ph = Po = None
        if with_preds:
            Ph = torch.empty((nch_dev, npix), dtype=torch.complex128).pin_memory()
            Ph.copy_(m._pix(P).cpu())
            Po = torch.empty_like(Ph).pin_memory()
        m.iterate_host(Xh, Ph, Xo, Po)  # warm-up
        ctx.barrier()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        w0.record()
        for _ in range(e2e_steps):
            m.iterate_host(Xh, Ph, Xo, Po)
            Xh, Xo = Xo, Xh
            Ph, Po = Po, Ph
        w1.record()
        torch.cuda.synchronize()
        e2e_s = max(w0.elapsed_time(w1) / 1e3, time.perf_counter() - t0)
        out["e2e_s"] = ctx.reduce([e2e_s])[0]
        out["e2e_steps"] = e2e_steps
        out["e2e_bytes"] = (ncoef + (npix if with_preds else 0)) * nch_dev * 16
        out["e2e_with_preds"] = with_preds
        del Xh, Ph, Xo, Po
    if dump:
        out["outputs"] = {"state": sample_outputs(last[0]), "predictions": sample_outputs(m._pix(last[1]))}
    del m, outer, op, reg, X, P, last
    return out


def measure_single_chain(ctx, args, iters=500):
    """per-chain latency: ONE MYULA chain at the bench bandlimit, the iteration replayed as one CUDA graph
    (`MYULA.run`'s path for device noise) -- the "per chain" half of the BASELINE metric"""
    torch = ctx.torch
    from pxmcmc_b200 import device as D, sht
    from pxmcmc_b200.forward import SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams
    from pxmcmc_b200.prior import S2_Wavelets_L1

    L, B, J_min = args.L, args.B, args.J_min
    data = sht.inverse(synthetic_flm(L), L).ravel()
    data = data / np.sqrt(np.mean(np.abs(data) ** 2))
    op = SphericalWaveletTransformOperator(data, 1.0, "synthesis", L, B, J_min)
    prm = PxMCMCParams(nsamples=1, nburn=0, ngap=1, delta=1e-6, lmda=1e-6, mu=1.0, verbosity=0, track=[])
    reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 1e-6, L=L, B=B, J_min=J_min)
    m = MYULA(op, reg, prm, noise="device", seed=99)
    X = D.to_dev_c(np.random.default_rng(0).laplace(size=(1, op.nparams)))
    op.fuse_ring = not args.no_ring_fusion
    P = m._initial_preds(X)
    chain = m.capture(X, P, iterations=1)
    for _ in range(50):
        chain.step()
    torch.cuda.synchronize()
    per = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters // 5):
            chain.step()
        b.record()
        torch.cuda.synchronize()
        per.append(a.elapsed_time(b) / (iters // 5))
    ms_it = float(np.median(per))
    import ctypes as C

    from pxmcmc_b200 import _lib

    fam = (C.c_longlong * 4)()
    _lib.check(_lib.lib.pxm_wav_plan_table_bytes_by_family(op.transform._plan(1).h, fam))
    # stage times of the same iteration launched eagerly (library events around every launch)
    n = 200
    _lib.check(_lib.lib.pxm_profile_begin(16 * n + 64))
    x, p_ = chain._state_raw()
    x, p_ = x.clone(), p_.clone()
    for _ in range(n):
        x, p_ = m.iterate(x, p_)
    msk, cnt = (C.c_double * 3)(), (C.c_longlong * 3)()
    _lib.check(_lib.lib.pxm_profile_end(msk, cnt))
    gram = C.c_longlong(0)
    _lib.check(_lib.lib.pxm_wav_plan_gram_bytes(op.transform._plan(1).h, C.byref(gram)))
    kind = P.kind if hasattr(P, "kind") else "pixels"
    chain.release()
    del chain, m, op
    if kind == "harm":  # the kappa-weighted W_j in both directions and the Gram table in between
        streamed = 2 * int(fam[1]) + int(gram.value)
    else:  # Lambda_L and the kappa-weighted W_j, once for Psi and once for Psi^dagger
        streamed = 2 * int(fam[0] + fam[1])
    return {"iterations_per_s": 1e3 / ms_it, "ms_per_iteration": ms_it, "iterations_timed": iters,
            "mode": "one chain, iteration replayed as one CUDA graph (in-place state), Philox noise; median of 5 blocks",
            "predictions": kind,
            "eager_stage_us": {"legendre": msk[0] / n * 1e3, "ring_fft": msk[1] / n * 1e3, "elementwise": msk[2] / n * 1e3},
            "table_bytes_streamed_per_iteration": streamed,
            "legendre_table_stream_GBps": streamed / (msk[0] / n / 1e3) / 1e9 if msk[0] > 0 else None,
            "note": f"{int(sum(cnt)) // n} launches per iteration: at one chain every kernel is a single short wave whose duration is its "
                    "own load-latency chain (ncu: long_scoreboard 59 % in the one-chain ring FFT), not a throughput limit"}


def measure_configs(ctx, args):
    """the BASELINE.json configurations that are parity-test cases (tests/test_gpu_configs.py) timed on one GPU:
    config 1 (MYULA L=32), config 2 (PxMALA, analysis prior, L=256), config 3 (SKROCK s=10, great-circle CSR, L=128)"""
    torch = ctx.torch
    from pxmcmc_b200 import _lib, device as D, paths, sht
    from pxmcmc_b200.forward import PathIntegralOperator, SphericalWaveletTransformOperator
    from pxmcmc_b200.mcmc import MYULA, PxMALA, SKROCK, PxMCMCParams
    from pxmcmc_b200.prior import L1, S2_Wavelets_L1, S2_Wavelets_L1_Power_Weights

    def data_map(L):
        d = sht.inverse(synthetic_flm(L), L).ravel()
        return d / np.sqrt(np.mean(np.abs(d) ** 2))

    def timed(fn, n, warm=10):
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

    out = {}
    # config 1
    L, B = 32, 1.5
    op = SphericalWaveletTransformOperator(data_map(L), 1.0, "synthesis", L, B, 2)
    prm = PxMCMCParams(delta=1e-6, lmda=1e-6, mu=1.0, verbosity=0, nsamples=1, track=[])
    reg = S2_Wavelets_L1("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 1e-6, L=L, B=B, J_min=2)
    m = MYULA(op, reg, prm, noise="device")
    X = D.to_dev_c(np.random.default_rng(0).laplace(size=(1, op.nparams)))
    chain = m.capture(X, D.to_dev_c(op.forward(X)), iterations=1)
    ms_it = timed(chain.step, 2000)
    chain.release()
    out["config1_myula_L32"] = {"ms_per_iteration": ms_it, "iterations_per_s": 1e3 / ms_it, "mode": "CUDA graph replay"}
    # config 2
    L, B = 256, 1.5
    op = SphericalWaveletTransformOperator(data_map(L), 0.1, "analysis", L, B, 2)
    prm = PxMCMCParams(delta=1e-7, lmda=1e-6, mu=1.0, verbosity=0, nsamples=5, nburn=0, ngap=100, track=["logposterior"])
    reg = L1("analysis", op.transform.inverse, op.transform.inverse_adjoint, 1e-6)
    PxMALA(op, reg, PxMCMCParams(delta=1e-7, lmda=1e-6, mu=1.0, verbosity=0, nsamples=1, nburn=0, ngap=1, track=[]),
           tune_delta=True, noise="device", seed=3).run(np.zeros(op.nparams))  # plans, tables
    m = PxMALA(op, reg, prm, tune_delta=True, noise="device", seed=3)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        m.run(np.zeros(op.nparams))
    torch.cuda.synchronize()
    nit = len(m.acceptance_trace)
    dt = (time.perf_counter() - t0) / nit
    out["config2_pxmala_analysis_L256"] = {"ms_per_iteration": dt * 1e3, "iterations_per_s": 1 / dt, "iterations": nit,
                                           "acceptance": float(np.mean(m.acceptance_trace)),
                                           "mode": "device-resident loop (accept test, step-size tuning, traces on the device), CUDA graph, "
                                                   "wall clock of run() incl. the host reads on the thinning grid"}
    del m, op, reg
    # config 3
    L, B, s = 128, 2, 10
    rng = np.random.default_rng(7)
    z = rng.uniform(-1, 1, size=(10000, 2))
    lon = rng.uniform(-180, 180, size=(10000, 2))
    lat = np.degrees(np.arcsin(z))
    t0 = time.perf_counter()
    A, (ip_d, ix_d, v_d) = paths.get_path_matrix(np.stack([lat[:, 0], lon[:, 0]], 1), np.stack([lat[:, 1], lon[:, 1]], 1), L,
                                                 device_csr=True)
    t_raster = time.perf_counter() - t0
    truth = data_map(L).real
    y = A @ truth + 0.05 * rng.standard_normal(A.shape[0])
    op = PathIntegralOperator(A, y, np.full(A.shape[0], 0.05), "synthesis", L, B, 2)
    prm = PxMCMCParams(delta=1e-6, lmda=5e-7, mu=1.0, s=s, verbosity=0, nsamples=1, track=[])
    reg = S2_Wavelets_L1_Power_Weights("synthesis", op.transform.inverse, op.transform.inverse_adjoint, 5e-7, L=L, B=B, J_min=2, eta=1)
    mg = SKROCK(op, reg, prm, noise="device", seed=5)
    gr = mg.capture(D.to_dev_c(np.zeros((1, op.nparams))))
    ms_step = timed(gr.step, 100)
    # the path operator alone: warp-per-row CSR SpMV and its transpose, HBM roofline
    xv = D.to_dev_c(rng.standard_normal(A.shape[1]) + 1j * rng.standard_normal(A.shape[1]))
    yv = D.to_dev_c(rng.standard_normal(A.shape[0]) + 1j * rng.standard_normal(A.shape[0]))
    def kernel_ms(fn, n=300):
        """device time of the library kernel itself (CUDA events recorded by the library around its launch)"""
        import ctypes as C

        for _ in range(10):
            fn()
        _lib.check(_lib.lib.pxm_profile_begin(n + 8))
        for _ in range(n):
            fn()
        msk, cnt = (C.c_double * 3)(), (C.c_longlong * 3)()
        _lib.check(_lib.lib.pxm_profile_end(msk, cnt))
        return msk[2] / max(cnt[2], 1)

    ms_f = kernel_ms(lambda: op.measurement.forward(xv))
    ms_t = kernel_ms(lambda: op.measurement.adjoint(yv))
    nbytes = A.nnz * 12 + 16 * (A.shape[0] + A.shape[1]) + 4 * A.shape[0]
    out["config3_skrock_pathintegral_L128"] = {
        "ms_per_step": ms_step, "steps_per_s": 1e3 / ms_step, "gradient_evaluations_per_step": s, "mode": "one CUDA graph per step",
        "path_matrix": {"shape": list(A.shape), "nnz": int(A.nnz), "rasterise_s": t_raster,
                        "built_by": "pxm_gc_rasterise: 10^4 great circles between random end points (seed 7), 160 points/rad"},
        "spmv": {"forward_us": ms_f * 1e3, "adjoint_us": ms_t * 1e3, "algorithmic_bytes": int(nbytes),
                 "forward_GBps": nbytes / (ms_f / 1e3) / 1e9, "adjoint_GBps": nbytes / (ms_t / 1e3) / 1e9,
                 "note": "nnz (8 + 4) + 16 (rows + cols) + 4 rows bytes; the matrix (11 MB) and both vectors are L2-resident "
                         "between launches, so this is launch-latency / L2 bound, not an HBM stream"}}
    del mg, gr, op, reg
    return out


def dgemm_peak(torch):
    """FP64 peak for the Legendre roofline: cuBLAS DGEMM measured right here (MEASURED_PEAKS.json has no FP64 entry)"""
    n = 6144
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    best = 1e9
    for _ in range(4):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        torch.matmul(a, b)
        s1.record()
        torch.cuda.synchronize()
        best = min(best, s0.elapsed_time(s1))
    return 2.0 * n ** 3 / best / 1e9  # TFLOP/s


def hbm_peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy bandwidth)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback stated in B200_PROFILING.md (MEASURED_PEAKS.json absent)"


def run_ours(args):
    ctx = Ctx()
    torch = ctx.torch
    L, B, J_min, nch = args.L, args.B, args.J_min, args.chains
    world = ctx.world
    main = measure_chains(ctx, args, nch, nch * world, args.steps, blocks=args.blocks, block_iters=args.block_iters,
                          e2e_steps=max(1, min(args.steps, args.e2e_steps)), dump=bool(args.dump_outputs) and ctx.rank == 0)
    release_plans()
    if "outputs" in main:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in main.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    extras = {}
    if not args.no_extras and not args.no_real_pairs and nch % 2 == 0:
        # the same sweep on REAL-valued data (the drivers' `_mw_` route): two real chains per complex device chain
        rp = measure_chains(ctx, args, nch, nch * world, args.steps, blocks=min(args.blocks, 3), block_iters=args.block_iters,
                            e2e_steps=max(1, min(args.steps, args.e2e_steps)), real=True)
        release_plans()
        ms_step = rp["ms"] / rp["steps"]
        extras["real_data_pairs"] = {
            "workload": f"{workload_name(L, B, J_min)} with REAL-valued data (experiments/earthtopography/main.py:83-85, the `_mw_` "
                        f"input route): MYULA(real_pairs=True), {nch} real chains per GPU as {nch // 2} complex device chains "
                        "(the linear operators of the synthesis path are complex-linear and real, so chain 2k rides in the real "
                        "and chain 2k+1 in the imaginary part; the reference carries every real chain as a complex array with "
                        "a zero imaginary part)",
            "value": world * nch * rp["steps"] / (rp["ms"] / 1e3), "unit": UNIT, "ms_per_step": ms_step, "steps": rp["steps"],
            "stage_ms_per_step": rp["stage_ms"], "gpu_launches": rp["launches"], "finite": rp["finite"],
            "predictions": rp.get("pred_kind"),
            "e2e": {"value": world * nch * rp["e2e_steps"] / rp["e2e_s"], "unit": UNIT, "h2d_bytes_per_step": rp["e2e_bytes"],
                    "d2h_bytes_per_step": rp["e2e_bytes"], "steps": rp["e2e_steps"],
                    "api": "MYULA(real_pairs=True).engine.iterate_host on the packed host state (16 B per PAIR of real coefficients)"},
            "parity": "tests/test_gpu_configs.py::test_config5_real_chain_pairs_L256 (every real chain against its own oracle "
                      "iteration, <= 1e-10), tests/test_gpu_samplers.py::test_real_chain_pairs_*"}
        if "sustained_ms_per_step" in rp:
            extras["real_data_pairs"]["sustained"] = {"value": world * nch / (rp["sustained_ms_per_step"] / 1e3), "unit": UNIT,
                                                      "ms_per_step": rp["sustained_ms_per_step"]}
    if world == 1 and not args.no_extras and not args.no_ring_fusion:
        # the reference's literal composition (predictions as pixels: 4 ring-FFT stages, 4 Legendre contractions per
        # iteration) measured in the same run, for comparison with the carried form of `value`
        a2 = argparse.Namespace(**vars(args))
        a2.no_ring_fusion = True
        lit = measure_chains(ctx, a2, nch, nch * world, args.steps)
        release_plans()
        extras["literal_composition"] = {"value": world * nch * lit["steps"] / (lit["ms"] / 1e3), "unit": UNIT,
                                         "ms_per_step": lit["ms"] / lit["steps"], "stage_ms_per_step": lit["stage_ms"],
                                         "gpu_launches": lit["launches"],
                                         "note": "same workload, predictions carried as pixels (--no-ring-fusion)"}
    if world > 1 and not args.no_extras:
        # config 5 as BASELINE.json words it: 64 chains in TOTAL, 64/N per GPU (strong scaling of the chain sweep)
        total = args.strong_total
        if total % world == 0:
            st = measure_chains(ctx, args, total // world, total, args.steps, blocks=3, block_iters=args.block_iters)
            release_plans()
            ms_step = st.get("sustained_ms_per_step", st["ms"] / st["steps"])
            extras["config5_strong"] = {
                "workload": f"{total} MYULA chains in total at L={L} B={B}, {total // world} per GPU, no data-path collective",
                "value": total / (ms_step / 1e3), "unit": UNIT, "scaling": "strong", "chains_per_gpu": total // world,
                "ms_per_step": ms_step, "stage_ms_per_step_max_over_ranks": st["stage_ms"], "finite": st["finite"]}
    if not args.no_extras:
        # config 4: one weak-lensing chain at L=512 m-sharded over the GPUs of this launch (strong scaling)
        a4 = argparse.Namespace(**vars(args))
        a4.L, a4.B, a4.steps, a4.warmup = 512, 2.0, max(args.steps, 100), 3
        wl = measure_msharded(ctx, a4, e2e=False)
        release_plans()
        if wl is not None:
            extras["config4_msharded"] = {k: wl[k] for k in ("metric", "value", "unit", "n_gpus", "ms_per_step", "scaling", "config",
                                                            "eager_ms_per_step", "stage_ms_per_step_max_over_ranks", "roofline",
                                                            "finite", "peer_barrier_ok", "launch_mode", "nvlink")}
    if ctx.rank == 0:
        if world == 1 and not args.no_extras:
            extras["per_chain_latency"] = measure_single_chain(ctx, args)
            release_plans()
            extras["configs"] = measure_configs(ctx, args)
            release_plans()
        peak = dgemm_peak(torch)
        hbm_peak, hbm_src = hbm_peak_gbs()
        traffic, tsrc = load_traffic()
        default_wl = (L, B, J_min, nch) == (256, 1.5, 2, 64)
        ncoef, npix, steps = main["ncoef"], main["npix"], main["steps"]
        ms = main["ms"]
        flops_step = algorithmic_flops_per_chain_iteration(L, B, J_min) * nch  # SURVEY 8(d): what the iteration is credited with
        # flops of the contractions actually executed: in the harmonic (Gram) form the two full-L contractions
        # (8 L^3 per chain) are replaced by one with G^m: 4 flops x sum_m (L-|m|)^2 entries
        exec_flops_step = flops_step
        if main.get("pred_kind") == "harm":
            gram_entries = L * L + 2 * sum((L - m) ** 2 for m in range(1, L))
            exec_flops_step = flops_step - nch * 8.0 * L ** 3 + nch * 4.0 * gram_entries
        st = main["stage_ms"]
        leg_tf = exec_flops_step / (st["legendre"] / 1e3) / 1e12 if st["legendre"] > 0 else None
        # ring FFT stages executed per step: coefficient side in and out, plus -- unless the predictions are carried as
        # ring coefficients -- pixel side in and out; every stage moves 16 B per sample on each of its two sides
        fft_bytes_step = 2 * 32.0 * (ncoef + (0 if main["ring_mode"] else npix)) * nch
        fft_stages = 2 if main["ring_mode"] else 4
        fft_gbs = fft_bytes_step / (st["ring_fft"] / 1e3) / 1e9 if st["ring_fft"] > 0 else None
        roof_fft = {"bound": "hbm", "kernel": "pxm_ring_fft3_kernel (persistent TMA-staged two-pass Bluestein ring FFT) + pxm_ring_fft2_kernel<.,0> "
                                              "for lengths <= 256: one launch of each per stage",
                    "achieved": fft_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": (fft_gbs / hbm_peak) if fft_gbs else None,
                    # dram__bytes_read + dram__bytes_write per stage (mean of the 4 stages of one step), from the tracked ncu summary
                    "traffic": (fft_stage_traffic(traffic, main["ring_mode"]) if default_wl else None),
                    "launches_timed": main["counts"][1], "algorithmic_bytes_per_stage": fft_bytes_step / fft_stages,
                    "stages_per_step": fft_stages,
                    "ms_per_step": st["ring_fft"], "peak_source": hbm_src,
                    "note": "HBM class per SURVEY 8(d): algorithmic bytes = pixels or coefficients in + ring coefficients out = "
                            "32 B x coefficients (and pixels, when the pixel side is not carried in ring / harmonic form) per stage per "
                            "chain.  DRAM traffic = algorithmic bytes and HBM is ~20-25 % busy: Bluestein (odd ring length 2l-1 = two "
                            "power-of-two FFTs of length >= 2n) needs 255 registers per thread, so an SM holds 8 warps and the kernel "
                            "is bound by exposed latency, not by HBM nor by FP64 issue (ablation builds, DESIGN.md section 3)"}
        roof_leg = {"bound": "tensor", "achieved": leg_tf, "peak": peak, "unit": "TFLOP/s", "frac": (leg_tf / peak) if leg_tf else None,
                    "traffic": traffic.get("legendre_bytes_per_launch") if default_wl else None,
                    "kernel": "pxm_legendre_kernel (FP64 DMMA)", "launches_timed": main["counts"][0],
                    "launches_per_step": main["counts"][0] / steps,
                    "executed_algorithmic_flops_per_step": exec_flops_step, "credited_flops_per_step_survey_8d": flops_step,
                    "ms_per_step": st["legendre"],
                    "note": "achieved = flops of the contractions executed / device time; with the Gram form of the pixel side "
                            "(one contraction with G^m = (2L-1) Lambda^T Lambda instead of the two full-L contractions) fewer flops are "
                            "executed than SURVEY 8(d) credits: against the credited figure the stage runs at "
                            f"{flops_step / (st['legendre'] / 1e3) / 1e12 if st['legendre'] > 0 else 0:.1f} TFLOP/s",
                    "peak_source": "cuBLAS DGEMM 6144^3 measured in this run (MEASURED_PEAKS.json has no FP64 figure)"}
        # `roofline` = the dominant kernel BY TIME of this run
        fft_dominant = st["ring_fft"] >= st["legendre"]
        line = {
            "metric": METRIC, "value": world * nch * steps / (ms / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(L, B, J_min),
                       "implementation": f"{nch} independent chains per GPU as one batch (per-chain it/s = value/(n_gpus*chains))",
                       "chains_per_gpu": nch, "ncoefs": ncoef, "npix": npix, "noise": "Philox4x32-10 in-kernel",
                       "predictions": ({"harm": "harmonic coefficients f_lm of the image: the pixel-side ring-FFT pair of consecutive iterations "
                                                "cancels and, the inverse covariance being one constant, the two full-L Legendre contractions "
                                                "collapse into one with the Gram matrix; pixels on demand (tracked samples)",
                                        "ring": "ring-Fourier coefficients of the image (the pixel-side ring-FFT pair of consecutive iterations "
                                                "cancels); pixels on demand"}.get(main.get("pred_kind"), "pixels")),
                       "l2_note": f"inputs larger than L2: per-step working set {(ncoef + npix) * nch * 16 * 3 / 2**20:.0f} MiB of state + "
                                  f"{main['table_bytes'] / 2**20:.0f} MiB of Legendre tables exceeds the 126 MB L2"},
            "per_chain_iterations_per_s": steps / (ms / 1e3),
            "gpu_launches": main["launches"], "finite": main["finite"],
            "stage_ms_per_step": st,
            "roofline": dict(roof_fft if fft_dominant else roof_leg, dominant_by_time=True),
            "roofline_ring_fft" if not fft_dominant else "roofline_legendre": roof_leg if fft_dominant else roof_fft,
            "traffic_source": tsrc,
            "e2e": {"value": world * nch * main["e2e_steps"] / main["e2e_s"], "unit": UNIT, "h2d_bytes_per_step": main["e2e_bytes"],
                    "d2h_bytes_per_step": main["e2e_bytes"], "steps": main["e2e_steps"],
                    "api": ("MYULA.iterate_host(X, preds): pinned host state + predictions -> device -> one iteration -> host, "
                            if main.get("e2e_with_preds") else
                            "MYULA.iterate_host(X): pinned host state -> device -> one iteration (the predictions behind the gradient "
                            "are recomputed from the state on the device) -> new state to the host, ") +
                           "chain groups pipelined over three streams (H2D | kernels | D2H); PCIe-bound" +
                           ("; all ranks share the host's PCIe / memory bandwidth (one NUMA node): this figure does not scale with N" if world > 1 else "")},
            "clocks": main["clocks"],
            "host_cpus_rank0": f"{ctx.cpus[0]}-{ctx.cpus[-1]} ({len(ctx.cpus)})" if ctx.cpus else None,
        }
        if "sustained_ms_per_step" in main:
            line["sustained"] = {"value": world * nch / (main["sustained_ms_per_step"] / 1e3), "unit": UNIT,
                                 "ms_per_step": main["sustained_ms_per_step"], "blocks": args.blocks, "iterations_per_block": args.block_iters,
                                 "blocks_ms_per_step": main["sustained_blocks_ms_per_step"],
                                 "note": "median over blocks of the max over ranks; the K-step `value` above is the contract's timed region"}
        line.update(extras)
        if not args.no_cpu_baseline and world == 1:
            os.environ["PXM_ORACLE_REPS"] = "4"  # ~13 s of CPU work at L=256
            t_it = _oracle_one_iteration((args.ref_L, B, J_min, 0))
            os.environ.pop("PXM_ORACLE_REPS")
            scale = algorithmic_flops_per_chain_iteration(L, B, J_min) / algorithmic_flops_per_chain_iteration(args.ref_L, B, J_min)
            line["cpu_baseline"] = {
                "value": 1.0 / (t_it * scale), "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"4 consecutive chain-iterations of the numpy oracle (port of the reference's Python layer over a numpy "
                          f"restatement of ssht / s2let; the real wheels are not installable here) at L={args.ref_L} ({t_it:.1f} s each on one core)"
                          + ("" if args.ref_L == L else f", scaled by the O(L^3) flop ratio {scale:.1f} to L={L}")}
        emit(line)
    ctx.close()


# ---------------------------------------------------------------------------------------
# config 4 of BASELINE.json: ONE weak-lensing chain at L=512, m-sharded over the GPUs (strong scaling)
# ---------------------------------------------------------------------------------------
def wl_mask(L):
    """equatorial band |90deg - theta| < 10deg plus the same band in a frame tilted by the
    ICRS->galactic pole angle (stand-in for utils.build_mask(L, 10), SURVEY.md 8d)"""
    th = (2 * np.arange(L) + 1) * np.pi / (2 * L - 1)
    ph = 2 * np.pi * np.arange(2 * L - 1) / (2 * L - 1)
    T, P = np.meshgrid(th, ph, indexing="ij")
    x, y, z = np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)
    a = np.radians(62.87)  # inclination of the galactic plane
    z2 = -np.sin(a) * y + np.cos(a) * z
    mask = np.ones((L, 2 * L - 1), dtype=bool)
    mask[np.abs(np.degrees(np.arcsin(np.clip(z, -1, 1)))) < 10] = False
    mask[np.abs(np.degrees(np.arcsin(np.clip(z2, -1, 1)))) < 10] = False
    return mask


def wl_flops_per_iteration(L, B, J_min):
    """SURVEY.md 8(d): 2 F_Psi + 2 F_SHT(L,0) + 2 F_SHT(L,2)"""
    return algorithmic_flops_per_chain_iteration(L, B, J_min) + 2 * 4.0 * L * L * L + 2 * 4.0 * L * (L * L - 4)


def nvlink_counters(local):
    """(tx, rx) bytes moved over all NVLink links of GPU `local` since boot, from NVML's throughput counters
    (NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX / _RX, KiB, all links); None when NVML does not expose them"""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        tx_id = getattr(pynvml, "NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX", 138)
        rx_id = getattr(pynvml, "NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX", 139)
        vals = pynvml.nvmlDeviceGetFieldValues(h, [(tx_id, 0xFFFFFFFF), (rx_id, 0xFFFFFFFF)])
        out = []
        for v in vals:
            if v.nvmlReturn != 0:
                return None
            out.append(float(v.value.ullVal) * 1024.0)
        return tuple(out)
    except Exception:  # noqa: BLE001
        return None


def measure_msharded(ctx, args, e2e=True):
    """-> the JSON line of the m-sharded weak-lensing workload on rank 0 (None elsewhere)"""
    import ctypes as C

    torch = ctx.torch
    world, rank = ctx.world, ctx.rank
    from pxmcmc_b200 import _lib, device as D
    from pxmcmc_b200 import msharded as ms
    from pxmcmc_b200.forward import ForwardOperator
    from pxmcmc_b200.mcmc import MYULA, PxMCMCParams

    L, B, J_min = args.L, args.B, args.J_min
    ex = ms.ProcessGroupExchange() if world > 1 else None
    tr = ms.ShardedSphericalWaveletTransform(L, B, J_min, rank, world, exchange=ex)
    mask = wl_mask(L)
    wl = ms.ShardedWeakLensing(L, rank, world, mask=mask, ngal=np.full((L, 2 * L - 1), 30.0), exchange=ex)
    rng = np.random.default_rng(11)  # same stream on every rank: full vectors, then sliced
    x_true = rng.laplace(size=tr.ncoefs_global) * 1e-3
    Xt = D.to_dev_c(tr.coef_layout.to_local(x_true))
    gdata = D.to_host(wl.forward(tr.inverse(Xt)))
    gdata = gdata + (rng.standard_normal(wl.ndata_global) + 1j * rng.standard_normal(wl.ndata_global))[wl.data_index]
    op = ForwardOperator(gdata, 1.0 / wl.inv_cov, "synthesis", transform=tr, measurement=wl, nparams=tr.ncoefs)
    if world > 1:
        op._pxm_allreduce = ms.allreduce_sum()
    # lmda = delta/2 as in experiments/weaklensing/main.py:114-115; delta small enough for the
    # unadjusted chain to stay stable on this synthetic data (the reference's driver runs PxMALA with tuning)
    prm = PxMCMCParams(delta=2e-12, lmda=1e-12, mu=1.0, verbosity=0, nsamples=1, nburn=0, ngap=1, track=[])
    reg = ms.sharded_s2_wavelets_l1(tr, prm.lmda * prm.mu, L, B, J_min)
    m = MYULA(op, reg, prm, noise="device", seed=4321, stream0=rank)
    X = D.to_dev_c(np.zeros((1, op.nparams)))
    P = D.to_dev_c(op.forward(X))

    for _ in range(max(args.warmup, 3)):
        X, P = m.iterate(X, P)
    # the GPU leaves its idle clocks only after some tens of ms of load: a fixed, rank-independent
    # number of extra untimed iterations (the ranks must issue identical call sequences)
    for _ in range(200):
        X, P = m.iterate(X, P)
    ctx.barrier()
    sampler = ClockSampler(ctx.local)
    sampler.start()
    steps = args.steps
    l0 = _lib.lib.pxm_launch_count()
    _lib.check(_lib.lib.pxm_profile_begin(32 * steps + 64))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record()
    for _ in range(steps):
        X, P = m.iterate(X, P)
    e1.record()
    ctx.barrier()
    ms_total = e0.elapsed_time(e1)
    ms_kind = (C.c_double * 3)()
    cnt_kind = (C.c_longlong * 3)()
    _lib.check(_lib.lib.pxm_profile_end(ms_kind, cnt_kind))
    launches = _lib.lib.pxm_launch_count() - l0
    sampler.stop_flag = True
    sampler.join(timeout=2)
    # ---- the same iteration replayed as ONE CUDA graph per rank (the product path for single chains:
    # ~36 launches + 12 peer barriers per iteration are launch-latency bound when issued one by one)
    eager_ms = ms_total
    chain = m.capture(X, P, iterations=1)
    nv0 = nvlink_counters(ctx.local)  # BEFORE the warm-up replays: nothing may idle the GPU between warm-up and timing
    nwarm = 20
    for _ in range(nwarm):
        chain.step()
    ctx.barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(steps):
        chain.step()
    g1.record()
    ctx.barrier()
    nv1 = nvlink_counters(ctx.local)
    ms_total = g0.elapsed_time(g1)
    nvl = [(nv1[0] - nv0[0]) / (steps + nwarm), (nv1[1] - nv0[1]) / (steps + nwarm)] if (nv0 and nv1) else [-1.0, -1.0]
    nvl = ctx.reduce(nvl, op="sum")  # bytes per iteration over all ranks (negative: counters unavailable)
    X, P = chain.state()
    ok = tr.plan.barrier_ok() and wl.s0.barrier_ok() and wl.s2.barrier_ok()
    lp, l2, pr = m._logpi_dev(X, P)
    ms_total, leg_ms, fft_ms, el_ms, bad, eager_ms = ctx.reduce([ms_total, ms_kind[0], ms_kind[1], ms_kind[2], 0.0 if ok else 1.0, eager_ms])
    # Legendre tables streamed per iteration (harmonic-space composition of Phi o Psi, SURVEY 3.5): the kappa_j-weighted
    # quadrature tables W_j of the wavelet plan for Psi and again for Psi^dagger, the spin-2 Lambda table (half of
    # that SHT plan) for Phi and again for Phi^dagger; the wavelet plan's Lambda_L and the spin-0 plan are never read
    fam = (C.c_longlong * 4)()
    _lib.check(_lib.lib.pxm_wav_plan_table_bytes_by_family(tr.plan.h, fam))
    fused = op._fused()
    tab_bytes = 2 * fam[1] + wl.s2.table_bytes if fused else 2 * (fam[0] + fam[1]) + wl.s0.table_bytes + wl.s2.table_bytes
    tab = ctx.reduce([float(tab_bytes)], op="sum")[0]

    e2e_val, nbytes = None, 0.0
    if e2e:
        # end to end: the chain state travels host -> device -> host around every iteration
        Xh, Ph = X.cpu().pin_memory(), P.cpu().pin_memory()
        Xo, Po = torch.empty_like(Xh).pin_memory(), torch.empty_like(Ph).pin_memory()
        m.iterate_host(Xh, Ph, Xo, Po)
        ctx.barrier()
        e2e_steps = max(1, min(steps, 20))
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            m.iterate_host(Xh, Ph, Xo, Po)
            Xh, Xo, Ph, Po = Xo, Xh, Po, Ph
        torch.cuda.synchronize()
        e2e_s = ctx.reduce([time.perf_counter() - t0])[0]
        nbytes = ctx.reduce([float((Xh.numel() + Ph.numel()) * 16)], op="sum")[0]
        e2e_val = e2e_steps / e2e_s
    chain.release()
    hbm_peak, hbm_src = hbm_peak_gbs()
    traffic, tsrc = load_traffic()
    line = None
    if rank == 0:
        flops = wl_flops_per_iteration(L, B, J_min)
        line = {
            "metric": f"MYULA iterations/s at L={L}, single weak-lensing chain, m-sharded", "value": steps / (ms_total / 1e3),
            "unit": "iterations/s", "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_total / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"config 4 of BASELINE.json: MYULA, spin-2 Kaiser-Squires weak-lensing operator (masked, ngal=30), "
                                   f"S2_Wavelets_L1, L={L} B={B} J_min={J_min}, ONE chain, azimuthal orders sharded over {world} GPU(s), "
                                   "theta<->m transposition fused into the Legendre contractions over NVLink peer memory",
                       "ncoefs": int(tr.ncoefs_global), "ndata": int(wl.ndata_global), "noise": "Philox4x32-10 in-kernel",
                       "l2_note": f"Legendre tables streamed per iteration: {tab / 2**20:.0f} MiB over all GPUs >> L2"},
            "gpu_launches": int(launches), "finite": bool(np.isfinite(lp).all() and abs(lp[0]) < 1e100), "peer_barrier_ok": bad == 0.0,
            "logposterior": float(np.real(lp[0])),
            "launch_mode": "one CUDA graph per iteration and rank (value); eager_ms_per_step = the same kernels launched one by one",
            "eager_ms_per_step": eager_ms / steps,
            "stage_ms_per_step_max_over_ranks": {"legendre": leg_ms / steps, "ring_fft": fft_ms / steps, "elementwise": el_ms / steps},
            "roofline": {"bound": "hbm", "kernel": "pxm_legendre_kernel (one right-hand side: table streaming bound)",
                         "achieved": tab * steps / (leg_ms / 1e3) / 1e9 if leg_ms > 0 else None,
                         "peak": world * hbm_peak, "unit": "GB/s", "peak_source": hbm_src,
                         # dram__bytes_read+write summed over the 4 Legendre launches of one iteration at N=1 (tracked ncu summary)
                         "traffic": traffic.get("wl_legendre_bytes_per_iteration") if (L, B, J_min, world) == (512, 2.0, 2, 1) and fused else None,
                         "note": "per ITERATION (4 launches): algorithmic bytes = every Legendre table the iteration uses, read once "
                                 "(sum over GPUs); with ONE right-hand side the contraction is a table stream, not DMMA-bound; "
                                 f"algorithmic flops {flops:.3e} per iteration -> {flops * steps / (leg_ms / 1e3) / 1e12 if leg_ms > 0 else 0:.2f} TFLOP/s aggregate"},
            "traffic_source": tsrc,
            "clocks": sampler.summary(),
        }
        # the theta <-> m transposition rides inside the Legendre kernels (peer stores / bulk pulls): NVML's link counters
        # around the timed region are the evidence of what actually crossed NVLink (no separate collective exists to count)
        npix_t, nscale_px = L * (2 * L - 1), int(tr.ncoefs_global)
        line["nvlink"] = {"tx_bytes_per_iteration_all_gpus": nvl[0] if nvl[0] >= 0 else None,
                          "rx_bytes_per_iteration_all_gpus": nvl[1] if nvl[1] >= 0 else None,
                          "source": "NVML NVLINK_THROUGHPUT_DATA_TX/RX (all links), difference around the graph replays, summed over ranks; null = NVML "
                                    "answers NOT_SUPPORTED in this VM (nvidia-smi nvlink -gt d prints N/A: gpurun_out/nvlink_probe.log), and ncu may not "
                                    "wrap a multi-rank command, so the expected figure below is the plan's own count",
                          "expected_bytes_per_iteration": (16.0 * (2 * npix_t + 2 * nscale_px) * (world - 1) / world) if world > 1 else 0.0,
                          "expected_note": "ring-Fourier slabs of one iteration: 2 spin-2 SHTs at L (16 B x L(2L-1) each) and the two "
                                           "multi-scale wavelet stages (16 B x ncoefs each), of which a share (N-1)/N changes rank"}
        if e2e_val is not None:
            line["e2e"] = {"value": e2e_val, "unit": "iterations/s", "h2d_bytes_per_step": int(nbytes), "d2h_bytes_per_step": int(nbytes),
                           "steps": e2e_steps, "api": "MYULA.iterate_host on every rank's local rows (pinned host buffers)"}
        if line["roofline"]["achieved"]:
            line["roofline"]["frac"] = line["roofline"]["achieved"] / line["roofline"]["peak"]
    del chain, m, op, reg, tr, wl
    return line


def run_msharded(args):
    ctx = Ctx()
    line = measure_msharded(ctx, args)
    if line is not None:
        emit(line)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chains", type=int, default=64, help="independent chains per GPU")
    ap.add_argument("--L", type=int, default=L_DEF)
    ap.add_argument("--B", type=float, default=B_DEF)
    ap.add_argument("--J_min", type=int, default=JMIN_DEF)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--blocks", type=int, default=5, help="sustained-rate blocks after the K-step timed region (0: none)")
    ap.add_argument("--block-iters", type=int, default=100)
    ap.add_argument("--strong-total", type=int, default=64, help="chains in TOTAL of the strong-scaling split (config 5)")
    ap.add_argument("--no-ring-fusion", action="store_true", help="carry the predictions as pixels (the reference's literal composition)")
    ap.add_argument("--no-real-pairs", action="store_true", help="skip the real-data / packed-chain-pairs leg (key `real_data_pairs`)")
    ap.add_argument("--e2e-with-preds", action="store_true", help="end-to-end leg: move the pixel-space predictions over PCIe too (round 1's form)")
    ap.add_argument("--no-extras", action="store_true", help="only the headline workload (no per-chain / config 1-4 / strong-split legs)")
    ap.add_argument("--ref-L", type=int, default=256, help="bandlimit of the bounded CPU sample")
    ap.add_argument("--ref-procs", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="chains", choices=["chains", "wl-msharded"],
                    help="chains: the BASELINE metric (independent chains, weak scaling); wl-msharded: config 4, one "
                         "weak-lensing chain m-sharded over the GPUs (strong scaling; defaults L=512 B=2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0's chains) to DIR/state.npy and DIR/predictions.npy: "
                         "float64 [k, 2] real and imaginary parts of the new chain states and of their pixel predictions, "
                         "each cut to a fixed sample of 2^20 elements when larger (sample_outputs); the inputs are the "
                         "same in every run with the same arguments")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "chains"):
        ap.error("--dump-outputs applies to the chains workload of --impl ours")
    # stdout carries exactly ONE JSON line: everything else this process prints (the samplers' "DONE", progress lines,
    # library banners) goes to stderr; emit() writes the line to the real stdout
    global _REAL_STDOUT
    _REAL_STDOUT = sys.stdout
    sys.stdout = sys.stderr
    if args.workload == "wl-msharded":
        if args.L == L_DEF and args.B == B_DEF:
            args.L, args.B = 512, 2.0
        return run_msharded(args)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
