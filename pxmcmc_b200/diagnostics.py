"""Streaming posterior summaries and multi-chain convergence diagnostics (no counterpart in the reference, which is
single-chain and stores every tracked sample).

What is summarised is exactly what the tracked arrays would hold, per scalar component of every element: ``chain`` with
``complex=True``: real and imaginary part as two components; ``chain`` with ``complex=False`` and ``predictions``: the
real part only; ``real_pairs=True``: every packed part is its own logical chain.  Each chain takes its samples on the
tracking grid (PxMALA: the accepted grid samples), exactly ``nsamples`` of them.  With n = nsamples, m logical chains,
h = n // 2, b = max(1, isqrt(n)), a = n // b:

* per-chain mean and variance (ddof 1) over the chain's n samples; pooled mean and variance lambda^2 (ddof 1) over all
  m n samples, ``std`` = lambda;
* split-R-hat (BDA3): half-chains [0, h) and [n - h, n) (the middle sample of odd n belongs to neither half), M = 2m,
  B = h / (M - 1) sum (theta_k - theta)^2, W = mean s_k^2, V = (h - 1) / h W + B / h, R = sqrt(V / W); NaN when h < 2
  or W = 0;
* ESS by replicated batch means (Gupta & Vats, 2020): batches [k b, (k + 1) b), k < a; sigma^2 = b / (m a - 1)
  sum (Y_ck - Y)^2, ESS = m n lambda^2 / sigma^2, MCSE = sqrt(sigma^2 / (m n)); NaN when m a < 2 or sigma^2 = 0.

The device keeps running moments (``pxm_stats_accumulate`` on the tracking grid) and reduces them to partial records
(``pxm_stats_partials``); ``finalize`` combines the records of any number of chain groups (GPUs, calls) with Chan's
rule and applies the formulas above.

``rank_diagnostics`` works on STORED samples instead: the rank-normalised split-R-hat and the bulk and tail ESS of
Vehtari et al. (2021), which need every pooled value (``pxm_rank_diagnostics``, DESIGN.md 7b).
"""
import math
from collections import namedtuple

import numpy as np


def batch_shape(n):
    """(h, b, a): half-chain length, batch size and number of batches of n samples per chain"""
    b = max(1, math.isqrt(int(n)))
    return int(n) // 2, b, int(n) // b


class Summary:
    """Posterior summary of one target.  Real components: ``mean``, ``var``, ``std``, ``rhat``, ``ess``, ``mcse`` are
    [n], ``chain_mean`` and ``chain_var`` [nchains, n] (logical chains).  Complex chains: ``mean`` and ``chain_mean``
    are complex; ``var``, ``std``, ``rhat``, ``ess``, ``mcse`` and ``chain_var`` gain a leading axis of 2 (re, im)."""

    STATS = ("mean", "var", "std", "chain_mean", "chain_var", "rhat", "ess", "mcse")

    def __init__(self, nchains, nsamples, **stats):
        self.nchains, self.nsamples = int(nchains), int(nsamples)
        for k in self.STATS:
            setattr(self, k, stats.get(k))

    def as_dict(self):
        return {k: getattr(self, k) for k in self.STATS if getattr(self, k) is not None}

    def wavelet_maps(self, name, L, B, J_min):
        """statistic `name` ([..., n] over the wavelet coefficients) split into one MW (theta, phi) map per scale, as
        `uncertainty.wavelet_credible_interval_range` does"""
        return _wavelet_maps(getattr(self, name), name, L, B, J_min)


def _wavelet_maps(v, name, L, B, J_min):
    from .utils import _multires_bandlimits

    v = np.asarray(v)
    maps, start = [], 0
    for bl in _multires_bandlimits(L, B, J_min):
        length = bl * (2 * bl - 1)
        maps.append(v[..., start:start + length].reshape(v.shape[:-1] + (bl, 2 * bl - 1)))
        start += length
    if start != v.shape[-1]:
        raise ValueError(f"{name} has {v.shape[-1]} entries, the wavelet tiling {start}")
    return maps


def _chan(a, b):
    """Chan's combination of two (count, mean, M2) triples of arrays"""
    na, ma, qa = a
    nb, mb, qb = b
    nn = na + nb
    with np.errstate(invalid="ignore", divide="ignore"):
        wb = np.where(nn > 0, nb / np.where(nn > 0, nn, 1), 0.0)
        d = mb - ma
        m = np.where(na == 0, mb, np.where(nb == 0, ma, ma + d * wb))
        q = np.where(na == 0, qb, np.where(nb == 0, qa, qa + qb + d * d * (na * wb)))
    return nn, m, q


def combine(records):
    """one partial record [10, ...] from those of disjoint chain groups (Chan's rule, counts as weights)"""
    records = [np.asarray(r, dtype=np.float64) for r in records]
    out = records[0].copy()
    for r in records[1:]:
        for i in (0, 4, 7):
            n, m, q = _chan((out[i], out[i + 1], out[i + 2]), (r[i], r[i + 1], r[i + 2]))
            out[i], out[i + 1], out[i + 2] = n, m, q
        out[3] = out[3] + r[3]
    return out


def statistics(record, nsamples):
    """(mean, var, rhat, ess, mcse) from a combined partial record [10, ...]"""
    h, b, _ = batch_shape(nsamples)
    K, _, hM2, ssum, pn, pm, pM2, bn, _, bM2 = record
    with np.errstate(invalid="ignore", divide="ignore"):
        var = np.where(pn > 1, pM2 / (pn - 1), np.nan)
        W = np.where(K > 0, ssum / np.where(K > 0, K, 1), np.nan)
        Bv = h * hM2 / (K - 1)
        if h >= 2:
            V = (h - 1) / h * W + Bv / h
            rhat = np.where(W == 0, np.nan, np.sqrt(V / W))
        else:
            rhat = np.full_like(var, np.nan)
        s2 = b * bM2 / (bn - 1)
        bad = (bn < 2) | (s2 == 0)
        ess = np.where(bad, np.nan, pn * var / s2)
        mcse = np.where(bad, np.nan, np.sqrt(s2 / pn))
    return pm, var, rhat, ess, mcse


def finalize(partials_list, chain_arrays=True):
    """`Summary` of the partial records of one or several chain groups (dicts as `PxMCMC.summary_partials()` gives
    them, in global chain order: the per-chain arrays are concatenated in list order)"""
    partials_list = list(partials_list)
    if not partials_list:
        raise ValueError("finalize: no partial records")
    n = int(partials_list[0]["nsamples"])
    if any(int(p["nsamples"]) != n for p in partials_list):
        raise ValueError("finalize: the chain groups ran for different numbers of samples")
    rec = combine([p["record"] for p in partials_list])  # [10, ncomp, nelem]
    ncomp = rec.shape[1]
    mean, var, rhat, ess, mcse = statistics(rec, n)
    nchains = sum(int(p["nchains"]) for p in partials_list)
    cm = cv = None
    if chain_arrays and all(p.get("chain_mean") is not None for p in partials_list):
        cm = np.concatenate([np.asarray(p["chain_mean"]) for p in partials_list], axis=0)  # [m, ncomp, nelem]
        cv = np.concatenate([np.asarray(p["chain_var"]) for p in partials_list], axis=0)
    if ncomp == 1:
        mean, var, rhat, ess, mcse = mean[0], var[0], rhat[0], ess[0], mcse[0]
        cm = None if cm is None else cm[:, 0]
        cv = None if cv is None else cv[:, 0]
    else:  # complex chains: complex means, a leading (re, im) axis on everything else
        mean = mean[0] + 1j * mean[1]
        cm = None if cm is None else cm[:, 0] + 1j * cm[:, 1]
        cv = None if cv is None else np.moveaxis(cv, 1, 0)
    return Summary(nchains, n, mean=mean, var=var, std=np.sqrt(var), chain_mean=cm, chain_var=cv, rhat=rhat, ess=ess,
                   mcse=mcse)


class StreamingSummary:
    """Device accumulators of the targets one sampler summarises (`PxMCMC(summarise=...)`).  `targets`: {name: (n,
    nchains, mode)} with n the vector length, nchains the device chains and mode as in pxm_stats_accumulate."""

    def __init__(self, targets, nsamples):
        from . import device as D

        self.nsamples = int(nsamples)
        self.layout = {k: tuple(int(x) for x in v) for k, v in targets.items()}
        self.acc = {k: D.stats_accumulator(*v) for k, v in self.layout.items()}

    def push(self, target, x, j=0, d_j=None):
        from . import device as D

        D.stats_accumulate_dev(self.acc[target], x, self.layout[target][2], self.nsamples, j=j, d_j=d_j)

    def partials(self):
        """{target: partial dict} (one pxm_stats_partials launch per target)"""
        from . import device as D

        out = {}
        for k, (n, nch, mode) in self.layout.items():
            rec, cm, cv = D.stats_partials_dev(self.acc[k], n, nch, mode, self.nsamples)
            ncomp = rec.shape[1]
            m = cm.shape[0] // ncomp
            out[k] = {"record": D.to_host(rec), "chain_mean": D.to_host(cm).reshape(m, ncomp, n),
                      "chain_var": D.to_host(cv).reshape(m, ncomp, n), "nsamples": self.nsamples, "nchains": m}
        return out

    def state(self):
        """host copies of the accumulators (checkpoints)"""
        from . import device as D

        return {k: D.to_host(a) for k, a in self.acc.items()}

    def load(self, arrays):
        import torch

        for k, a in self.acc.items():
            src = np.asarray(arrays[k])
            if src.shape != tuple(a.shape):
                raise ValueError(f"checkpoint summary accumulator {k} has shape {src.shape}, expected {tuple(a.shape)}")
            a.copy_(torch.from_numpy(np.ascontiguousarray(src)))


def credible_tails(npooled, alpha):
    """(npooled, lo_a, gamma_a, lo_b, gamma_b): numpy's linear-quantile virtual indices of alpha / 2 and 1 - alpha / 2
    among npooled values, evaluated as `uncertainty.credible_interval_range` evaluates them"""
    from .uncertainty import _virtual_index

    N = int(npooled)
    return (N,) + _virtual_index(N, alpha / 2) + _virtual_index(N, 1 - alpha / 2)


class CredibleIntervals:
    """(1 - alpha) credible intervals of one target (`PxMCMC(credible=...)`): ``lower`` and ``upper`` are numpy's
    linear quantiles at alpha / 2 and 1 - alpha / 2 over the ``npooled`` = nchains * nsamples tracked samples of every
    element, pooled over the logical chains; ``range = upper - lower`` is what `uncertainty.credible_interval_range`
    gives for the stored samples.  Real components: [n]; complex chains: a leading axis of 2 (re, im)."""

    def __init__(self, alpha, nchains, nsamples, lower, upper):
        self.alpha, self.nchains, self.nsamples = float(alpha), int(nchains), int(nsamples)
        self.npooled = self.nchains * self.nsamples
        self.lower, self.upper = np.asarray(lower), np.asarray(upper)
        self.range = self.upper - self.lower

    def wavelet_maps(self, name, L, B, J_min):
        """`lower`, `upper` or `range` split into one MW (theta, phi) map per wavelet scale (`Summary.wavelet_maps`)"""
        return _wavelet_maps(getattr(self, name), name, L, B, J_min)


class StreamingCredible:
    """Device tail heaps of the targets one sampler bounds (`PxMCMC(credible=...)`).  `targets`: {name: (n, nchains,
    mode)} with n the vector length, nchains the device chains and mode as in pxm_credible_push (all targets of a
    sampler pool the same logical chains).  `count`: samples pooled per element so far."""

    def __init__(self, targets, nsamples, alpha):
        import torch

        from . import device as D

        self.layout = {k: tuple(int(x) for x in v) for k, v in targets.items()}
        _, nch, mode = next(iter(self.layout.values()))
        self.parts = 2 if mode == 2 else 1  # logical chains per device chain
        self.alpha, self.nsamples = float(alpha), int(nsamples)
        self.nchains = nch * self.parts
        self.tails = credible_tails(self.nchains * self.nsamples, self.alpha)
        need = sum(8 * D.credible_state_doubles(n, m, self.tails) for n, _, m in self.layout.values())
        free = torch.cuda.mem_get_info(D.dev())[0]
        if need > free:
            raise ValueError(f"credible: the tail heaps of {self.nchains} x {self.nsamples} pooled samples at alpha = "
                             f"{self.alpha} need {need} bytes of device memory, {free} are free (fewer samples or a "
                             f"larger alpha need less)")
        self.heaps = {k: D.credible_state(n, m, self.tails) for k, (n, _, m) in self.layout.items()}
        self.count = 0

    def push(self, samples, d_j=None, nactive=None):
        """one push per target of `samples` = {target: [nchains, n] device tensor}; `nactive`: chains with d_j >= 0
        (known on the host, so the pooled count needs no synchronisation); None: every chain"""
        from . import device as D

        for k, (_, nch, mode) in self.layout.items():
            D.credible_push_dev(self.heaps[k], samples[k], mode, self.tails, self.count, d_j)
        self.count += (nch if nactive is None else int(nactive)) * self.parts

    def intervals(self):
        """{target: CredibleIntervals} (one pxm_credible_finalize launch per target)"""
        from . import device as D

        if self.count != self.tails[0]:
            raise RuntimeError(f"credible: {self.count} of {self.tails[0]} samples pooled")
        out = {}
        for k, (n, _, mode) in self.layout.items():
            lo, hi = (D.to_host(a) for a in D.credible_finalize_dev(self.heaps[k], n, mode, self.tails))
            if mode != 1:
                lo, hi = lo[0], hi[0]
            out[k] = CredibleIntervals(self.alpha, self.nchains, self.nsamples, lo, hi)
        return out

    def state(self):
        """host copies of the heaps and the pooled count (checkpoints)"""
        from . import device as D

        d = {k: D.to_host(a) for k, a in self.heaps.items()}
        d["count"] = np.int64(self.count)
        return d

    def load(self, arrays):
        import torch

        for k, a in self.heaps.items():
            src = np.asarray(arrays[k])
            if src.shape != tuple(a.shape):
                raise ValueError(f"checkpoint credible heaps {k} have shape {src.shape}, expected {tuple(a.shape)}")
            a.copy_(torch.from_numpy(np.ascontiguousarray(src)))
        self.count = int(arrays["count"])


RankDiagnostics = namedtuple("RankDiagnostics", ["rhat", "ess_bulk", "ess_tail"])


def rank_diagnostics(chains, max_bytes=2 << 30):
    """Rank-normalised split-R-hat and bulk / tail ESS of every parameter of stored chains (Vehtari, Gelman, Simpson,
    Carpenter & Buerkner 2021; what ArviZ's rhat(method="rank") and ess(method="bulk" | "tail") report), on the GPU.

    :param chains: [nchains, nsamples, nparams] real array (a tracked ``chain`` / ``preds`` of a multi-chain sampler),
        or [nsamples, nparams] for one chain: numpy (``np.memmap`` included) or a float64 CUDA tensor.  Complex
        chains: pass ``.real`` and ``.imag`` separately.  nchains * nsamples <= 16 384.
    :param max_bytes: device memory of one block of columns (the block and its transposed copy); host arrays are
        uploaded block by block.
    :return: ``RankDiagnostics(rhat, ess_bulk, ess_tail)``, each [nparams], of the same kind as ``chains``.  All three
        are NaN for a parameter with a non-finite sample, and for every parameter when nsamples < 4."""
    from . import device as D
    from ._lib import lib

    on_dev = D.is_dev(chains)
    if on_dev:
        if chains.is_complex():
            raise TypeError("rank_diagnostics: complex chains; pass .real and .imag separately")
    else:
        chains = np.asarray(chains)
        if np.iscomplexobj(chains):
            raise TypeError("rank_diagnostics: complex chains; pass .real and .imag separately")
    if chains.ndim not in (2, 3):
        raise ValueError(f"rank_diagnostics: expected [nchains, nsamples, nparams] or [nsamples, nparams], got "
                         f"{chains.ndim} dimensions")
    m, n, npar = (1,) + tuple(chains.shape) if chains.ndim == 2 else tuple(chains.shape)
    S, limit = m * n, lib.pxm_quantile_columns_max_samples()
    if S > limit:
        raise ValueError(f"rank_diagnostics: {m} x {n} = {S} samples per parameter exceed the {limit} of the "
                         f"shared-memory sort")
    step = max(32, int(max_bytes // (16 * max(S, 1))) // 32 * 32)  # columns per block
    if on_dev:
        x = chains.reshape(S, npar).to(D.FDT)
        if npar > 1 and x.stride(1) != 1:
            x = x.contiguous()
        out = [x.new_empty(npar) for _ in range(3)]
        for c0 in range(0, npar, step):
            for o, r in zip(out, D.rank_diagnostics_dev(x[:, c0:c0 + step], m, n)):
                o[c0:c0 + step] = r
        return RankDiagnostics(*out)
    x = chains.reshape(S, npar)
    out = np.empty((3, npar))
    for c0 in range(0, npar, step):
        res = D.rank_diagnostics_dev(D.to_dev_f(x[:, c0:c0 + step]), m, n)
        for k in range(3):
            out[k, c0:c0 + step] = D.to_host(res[k])
    return RankDiagnostics(out[0], out[1], out[2])
