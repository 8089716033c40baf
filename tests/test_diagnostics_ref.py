"""CPU tests of the streaming posterior summaries: the two-pass oracle (oracle/diagnostics_ref.py) against hand-computed
values and known statistical behaviour, the host combine (`diagnostics.finalize`) of partial records from uneven chain
groups, the world_size-2 gloo gather of `sharding.gather_summary`, and the save / load round trip."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle import diagnostics_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _close(a, b, tol):
    a, b = np.asarray(a, dtype=complex), np.asarray(b, dtype=complex)
    assert a.shape == b.shape
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(a)
    assert np.all(np.abs(a[ok] - b[ok]) <= tol * np.maximum(1.0, np.abs(b[ok]))), (a, b)


def test_oracle_hand_computed_even_n():
    # m = 2, n = 4: h = 2, b = 2, a = 2 (halves and batches coincide)
    x = np.array([[0.0, 1, 2, 3], [1, 3, 5, 7]])
    s = R.summarise(x)
    # half means .5, 2.5, 2, 6 (grand mean 2.75, sum of squares 16.25); half variances .5, .5, 2, 2
    # B = 2/3 16.25, W = 1.25, V = W/2 + B/2 -> V/W = 29/6
    assert np.isclose(s["rhat"], np.sqrt(29 / 6), rtol=1e-15)
    # pooled: mean 2.75, sum of squares 37.5 -> var 37.5/7; sigma^2 = 2/3 16.25 = 65/6
    assert np.isclose(s["mean"], 2.75) and np.isclose(s["var"], 37.5 / 7, rtol=1e-15)
    assert np.isclose(s["ess"], 1800 / 455, rtol=1e-15) and np.isclose(s["mcse"], np.sqrt(65 / 48), rtol=1e-15)
    assert np.allclose(s["chain_mean"], [1.5, 4]) and np.allclose(s["chain_var"], [5 / 3, 20 / 3])


def test_oracle_hand_computed_odd_n_middle_sample():
    # m = 2, n = 5: h = 2 (the middle sample j = 2 is in neither half), b = 2, a = 2 (sample 4 is in no batch)
    x = np.array([[0.0, 1, 2, 3, 4], [0, 2, 4, 6, 8]])
    s = R.summarise(x)
    # half means .5, 3.5, 1, 7 (mean 3, squares 26.5); half variances .5, .5, 2, 2 -> V/W = 227/30
    assert np.isclose(s["rhat"], np.sqrt(227 / 30), rtol=1e-15)
    # batch means .5, 2.5, 1, 5 (mean 2.25, squares 12.25): sigma^2 = 49/6; pooled var 60/9
    assert np.isclose(s["var"], 20 / 3, rtol=1e-15) and np.isclose(s["mean"], 3.0)
    assert np.isclose(s["ess"], 400 / 49, rtol=1e-15) and np.isclose(s["mcse"], np.sqrt(49 / 60), rtol=1e-15)
    assert np.allclose(s["chain_mean"], [2, 4]) and np.allclose(s["chain_var"], [2.5, 10])
    # the host combine of the oracle's partial record gives the same numbers
    from pxmcmc_b200.diagnostics import finalize

    f = finalize([{"record": R.partial_record(x[:, :, None, None]), "nsamples": 5, "nchains": 2}])
    for k in ("mean", "var", "rhat", "ess", "mcse"):
        _close(getattr(f, k), np.atleast_1d(s[k]), 1e-14)


def test_iid_normal_rhat_and_ess():
    x = np.random.default_rng(0).standard_normal((8, 10_000, 4))
    s = R.summarise(x)
    assert np.all((s["rhat"] > 0.99) & (s["rhat"] < 1.01))
    r = s["ess"] / (8 * 10_000)
    assert np.all((r > 0.85) & (r < 1.15)), r


def test_ar1_ess():
    rho, m, n, k = 0.5, 8, 10_000, 16
    rng = np.random.default_rng(1)
    e = rng.standard_normal((m, n, k))
    x = np.empty_like(e)
    x[:, 0] = e[:, 0] / np.sqrt(1 - rho ** 2)
    for t in range(1, n):
        x[:, t] = rho * x[:, t - 1] + e[:, t]
    s = R.summarise(x)
    want = m * n * (1 - rho) / (1 + rho)
    assert abs(np.mean(s["ess"]) / want - 1) < 0.1, np.mean(s["ess"]) / want


def test_offset_chain_rhat():
    x = np.random.default_rng(2).standard_normal((4, 1000, 3))
    x[2] += 3.0
    assert np.all(R.summarise(x)["rhat"] > 1.5)


def test_nan_where_undefined():
    rng = np.random.default_rng(3)
    for n in (1, 2, 3):  # h < 2
        s = R.summarise(rng.standard_normal((3, n, 2)))
        assert np.all(np.isnan(s["rhat"]))
    s = R.summarise(np.ones((3, 10, 2)))  # constant chains: W = 0, sigma^2 = 0
    assert np.all(np.isnan(s["rhat"])) and np.all(np.isnan(s["ess"])) and np.all(np.isnan(s["mcse"]))
    s = R.summarise(rng.standard_normal((1, 1, 2)))  # one batch in all: m a < 2
    assert np.all(np.isnan(s["ess"])) and np.all(np.isnan(s["var"]))


@pytest.mark.parametrize("n", [1, 4, 7, 100])
def test_finalize_combines_uneven_chain_groups(n):
    """partial records of the chain groups {1, 31, 32} of 64 combine (Chan, weighted by counts) into the statistics of
    all 64 chains"""
    from pxmcmc_b200.diagnostics import finalize

    rng = np.random.default_rng(n)
    x = rng.standard_normal((64, n, 50)) * np.exp(rng.uniform(-2, 2, (64, 1, 1))) + rng.uniform(-5, 5, (64, 1, 1))
    groups, parts, c0 = (1, 31, 32), [], 0
    for g in groups:
        xs = x[c0:c0 + g]
        parts.append({"record": R.partial_record(xs[:, :, None, :]), "nsamples": n, "nchains": g,
                      "chain_mean": xs.mean(axis=1)[:, None], "chain_var": (xs.var(axis=1, ddof=1) if n > 1 else
                                                                            np.full((g, 50), np.nan))[:, None]})
        c0 += g
    f = finalize(parts)
    ref = R.summarise(x)
    assert f.nchains == 64 and f.nsamples == n
    for k in ("mean", "var", "std", "rhat", "ess", "mcse", "chain_mean", "chain_var"):
        _close(getattr(f, k), ref[k], 1e-12)


def test_finalize_complex_layout_and_wavelet_maps():
    from pxmcmc_b200.diagnostics import finalize
    from pxmcmc_b200.utils import _multires_bandlimits

    L, B, J = 10, 2, 2
    n = sum(bl * (2 * bl - 1) for bl in _multires_bandlimits(L, B, J))
    rng = np.random.default_rng(4)
    z = rng.standard_normal((3, 9, n)) + 1j * rng.standard_normal((3, 9, n))
    comp = np.stack([z.real, z.imag], axis=2)  # [m, n, 2, nelem]
    f = finalize([{"record": R.partial_record(comp), "nsamples": 9, "nchains": 3,
                   "chain_mean": comp.mean(axis=1), "chain_var": comp.var(axis=1, ddof=1)}])
    re, im = R.summarise(z.real), R.summarise(z.imag)
    _close(f.mean, re["mean"] + 1j * im["mean"], 1e-13)
    _close(f.chain_mean, re["chain_mean"] + 1j * im["chain_mean"], 1e-13)
    for k in ("var", "rhat", "ess", "mcse", "chain_var"):
        assert getattr(f, k).shape[0] == 2
        _close(getattr(f, k), np.stack([re[k], im[k]]), 1e-12)
    maps = f.wavelet_maps("var", L, B, J)
    assert [m.shape for m in maps] == [(2, bl, 2 * bl - 1) for bl in _multires_bandlimits(L, B, J)]
    assert np.array_equal(np.concatenate([m.reshape(2, -1) for m in maps], axis=1), f.var)


_WORKER = r"""
import os, sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, {root!r})
from oracle import diagnostics_ref as R
from pxmcmc_b200.sharding import chain_shard, gather_summary
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world, total, n = dist.get_rank(), dist.get_world_size(), 5, 11
x = np.random.default_rng(7).standard_normal((total, n, 6))
start, count = chain_shard(total, world, rank)
xs = x[start:start + count]
part = {{"chain": {{"record": R.partial_record(xs[:, :, None]), "nsamples": n, "nchains": count,
                    "chain_mean": xs.mean(axis=1)[:, None], "chain_var": xs.var(axis=1, ddof=1)[:, None]}}}}
out = gather_summary(part, total)
if rank == 0:
    ref = R.summarise(x)
    s = out["chain"]
    assert s.nchains == total
    for k in ("mean", "var", "rhat", "ess", "mcse", "chain_mean", "chain_var"):
        assert np.allclose(getattr(s, k), ref[k], rtol=1e-12, atol=0), k
    print("SUMMARY_OK")
else:
    assert out is None
dist.barrier()
dist.destroy_process_group()
"""


def test_gather_summary_gloo_world_size_2(tmp_path):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "summary_worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=180) for p in procs]
    for p, (o, e) in zip(procs, outs):
        assert p.returncode == 0, e[-2000:]
    assert "SUMMARY_OK" in outs[0][0]


@pytest.mark.parametrize("with_summary", [False, True])
def test_saving_roundtrip_with_and_without_summaries(tmp_path, with_summary):
    from pxmcmc_b200 import saving
    from pxmcmc_b200.diagnostics import finalize
    from pxmcmc_b200.mcmc import PxMCMCParams

    class Run:
        pass

    run = Run()
    run.logPi, run.chain = np.arange(4.0), np.arange(12.0).reshape(4, 3)
    x = np.random.default_rng(5).standard_normal((2, 6, 3))
    if with_summary:
        run.summary = {"chain": finalize([{"record": R.partial_record(x[:, :, None]), "nsamples": 6, "nchains": 2,
                                           "chain_mean": x.mean(axis=1)[:, None], "chain_var": x.var(axis=1, ddof=1)[:, None]}])}
    prm = PxMCMCParams(nsamples=4, nburn=1, ngap=2, track=["chain"])
    path = saving.save_mcmc(run, prm, str(tmp_path), filename="out", L=10)
    data, attrs = saving.load_mcmc(path)
    assert np.array_equal(data["chain"], run.chain) and int(attrs["L"]) == 10
    got = saving.summaries(data)
    if not with_summary:
        assert got == {} and sorted(data) == ["chain", "logposterior"]
        return
    s, ref = got["chain"], run.summary["chain"]
    assert (s.nchains, s.nsamples) == (2, 6)
    for k in ref.STATS:
        assert np.array_equal(getattr(s, k), getattr(ref, k), equal_nan=True), k
