"""Restatement of the streaming posterior summaries (pxmcmc_b200.diagnostics, DESIGN.md 7b) from FULL stored samples,
with two-pass numpy formulas (np.mean, np.var(ddof=1)).  Nothing here uses running moments: it is what the streaming
kernels are checked against.

samples: real array [m, n, ...] (m chains, n samples each, any trailing element shape).  With h = n // 2,
b = max(1, isqrt(n)), a = n // b:
  split-R-hat: half-chains [0, h) and [n - h, n) (the middle sample of odd n is in neither), M = 2m, B = h/(M-1)
  sum (theta_k - theta)^2, W = mean s_k^2, V = (h-1)/h W + B/h, R = sqrt(V/W); NaN when h < 2 or W = 0.
  ESS (replicated batch means): batches [k b, (k+1) b), k < a; sigma^2 = b/(m a - 1) sum (Y_ck - Y)^2,
  ESS = m n lambda^2 / sigma^2, MCSE = sqrt(sigma^2 / (m n)); NaN when m a < 2 or sigma^2 = 0.
"""
import math

import numpy as np


def batch_shape(n):
    """(h, b, a) of n samples per chain"""
    b = max(1, math.isqrt(n))
    return n // 2, b, n // b


def summarise(samples):
    x = np.asarray(samples, dtype=np.float64)
    m, n = x.shape[:2]
    h, b, a = batch_shape(n)
    nan = np.full(x.shape[2:], np.nan)
    flat = x.reshape((m * n,) + x.shape[2:])
    out = {"nchains": m, "nsamples": n, "mean": flat.mean(axis=0), "chain_mean": x.mean(axis=1)}
    with np.errstate(invalid="ignore", divide="ignore"):
        out["var"] = flat.var(axis=0, ddof=1) if m * n > 1 else nan.copy()
        out["chain_var"] = x.var(axis=1, ddof=1) if n > 1 else np.full((m,) + x.shape[2:], np.nan)
        out["std"] = np.sqrt(out["var"])
        if h >= 2:
            halves = np.concatenate([x[:, :h], x[:, n - h:]], axis=0)  # [2m, h, ...]
            hm = halves.mean(axis=1)
            M = halves.shape[0]
            Bv = h / (M - 1) * ((hm - hm.mean(axis=0)) ** 2).sum(axis=0)
            W = halves.var(axis=1, ddof=1).mean(axis=0)
            V = (h - 1) / h * W + Bv / h
            out["rhat"] = np.where(W == 0, np.nan, np.sqrt(V / W))
        else:
            out["rhat"] = nan.copy()
        if m * a >= 2:
            Y = x[:, : a * b].reshape((m, a, b) + x.shape[2:]).mean(axis=2).reshape((m * a,) + x.shape[2:])
            s2 = b / (m * a - 1) * ((Y - Y.mean(axis=0)) ** 2).sum(axis=0)
            out["ess"] = np.where(s2 == 0, np.nan, m * n * out["var"] / s2)
            out["mcse"] = np.where(s2 == 0, np.nan, np.sqrt(s2 / (m * n)))
        else:
            out["ess"], out["mcse"] = nan.copy(), nan.copy()
    return out


def partial_record(samples):
    """the 10-field partial record of pxm_stats_partials for these chains, two-pass: half-chain count, mean and M2 of
    the half-chain means, sum of the half-chain variances; sample count, mean, M2; batch count, mean and M2 of the
    batch means"""
    x = np.asarray(samples, dtype=np.float64)
    m, n = x.shape[:2]
    h, b, a = batch_shape(n)
    tail = x.shape[2:]
    rec = np.zeros((10,) + tail)
    if h >= 1:
        halves = np.concatenate([x[:, :h], x[:, n - h:]], axis=0)
        hm = halves.mean(axis=1)
        rec[0] = 2 * m
        rec[1] = hm.mean(axis=0)
        rec[2] = ((hm - rec[1]) ** 2).sum(axis=0)
        if h >= 2:
            rec[3] = halves.var(axis=1, ddof=1).sum(axis=0)
    flat = x.reshape((m * n,) + tail)
    rec[4] = m * n
    rec[5] = flat.mean(axis=0)
    rec[6] = ((flat - rec[5]) ** 2).sum(axis=0)
    Y = x[:, : a * b].reshape((m, a, b) + tail).mean(axis=2).reshape((m * a,) + tail)
    rec[7] = m * a
    rec[8] = Y.mean(axis=0)
    rec[9] = ((Y - rec[8]) ** 2).sum(axis=0)
    return rec
