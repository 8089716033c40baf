"""Saving an MCMC run, mirroring ``pxmcmc/saving.py`` of the reference: the tracked arrays become
datasets named ``logposterior, predictions, chain, L2s, priors, acceptances, deltas``, the runtime
parameters and any keyword arguments become attributes.

The reference writes HDF5 through h5py (pxmcmc/saving.py:18-36).  h5py is used when it can be
imported (same file, same names: the reference's plot scripts read it unchanged); otherwise the
same names go into ``<filename>.npz`` (datasets as arrays, attributes under ``attrs/<name>``) and
``load_mcmc`` reads either.

Streaming posterior summaries (``PxMCMC(summarise=...)``, an extension) are written, when present, as datasets
``summary/<target>/<statistic>`` (plus ``nchains`` and ``nsamples``); ``load_mcmc`` returns them under the same flat
names and ``summaries`` turns them back into ``diagnostics.Summary`` objects.  Streaming credible intervals
(``PxMCMC(credible=...)``) likewise go into ``credible/<target>/{lower,upper,range,alpha,nchains,nsamples}``, read back
by ``credible_intervals``."""
import os

import numpy as np

DATASETS = (("logPi", "logposterior"), ("preds", "predictions"), ("chain", "chain"), ("L2s", "L2s"), ("priors", "priors"),
            ("acceptance_trace", "acceptances"), ("deltas_trace", "deltas"))


def _collect(mcmc, params, kwargs):
    data = {}
    for attr, name in DATASETS:
        if hasattr(mcmc, attr):
            arr = np.asarray(getattr(mcmc, attr))
            data[name] = arr.astype("i1") if name == "acceptances" else arr
    for target, sm in (getattr(mcmc, "summary", None) or {}).items():
        for stat, arr in sm.as_dict().items():
            data[f"summary/{target}/{stat}"] = np.asarray(arr)
        data[f"summary/{target}/nchains"] = np.asarray(sm.nchains)
        data[f"summary/{target}/nsamples"] = np.asarray(sm.nsamples)
    for target, ci in (getattr(mcmc, "credible_intervals", None) or {}).items():
        for name in ("lower", "upper", "range", "alpha", "nchains", "nsamples"):
            data[f"credible/{target}/{name}"] = np.asarray(getattr(ci, name))
    attrs = {k: getattr(params, k) for k in params.__dict__.keys()}
    attrs.update(kwargs)
    return data, attrs


def save_mcmc(mcmc, params, outpath, filename="outputs", **kwargs):
    """Save the tracked arrays of ``mcmc`` (after ``run``) and the parameters ``params`` in
    ``outpath/filename.hdf5`` (h5py available) or ``outpath/filename.npz``; returns the path."""
    data, attrs = _collect(mcmc, params, kwargs)
    try:
        import h5py
    except ImportError:
        h5py = None
    if h5py is not None:
        path = os.path.join(outpath, f"{filename}.hdf5")
        with h5py.File(path, "w") as f:
            for name, arr in data.items():
                f.create_dataset(name, data=arr)
            for k, v in attrs.items():
                f.attrs[k] = v
        return path
    path = os.path.join(outpath, f"{filename}.npz")
    flat = dict(data)
    for k, v in attrs.items():
        flat[f"attrs/{k}"] = np.asarray(v)
    np.savez(path, **flat)
    return path


def load_mcmc(path):
    """(datasets, attrs) dictionaries of a file written by ``save_mcmc``"""
    if path.endswith(".npz"):
        with np.load(path, allow_pickle=False) as f:
            data = {k: f[k] for k in f.files if not k.startswith("attrs/")}
            attrs = {k[6:]: (f[k][()] if f[k].ndim == 0 else f[k]) for k in f.files if k.startswith("attrs/")}
        return data, attrs
    import h5py

    with h5py.File(path, "r") as f:
        data = {}
        f.visititems(lambda name, obj: data.__setitem__(name, obj[()]) if isinstance(obj, h5py.Dataset) else None)
        return data, dict(f.attrs)


def summaries(data):
    """{target: diagnostics.Summary} from the datasets `load_mcmc` returned (empty when the file has none)"""
    from .diagnostics import Summary

    out = {}
    for target in sorted({k.split("/")[1] for k in data if k.startswith("summary/")}):
        pre = f"summary/{target}/"
        stats = {k[len(pre):]: data[k] for k in data if k.startswith(pre)}
        out[target] = Summary(int(stats.pop("nchains")), int(stats.pop("nsamples")), **stats)
    return out


def credible_intervals(data):
    """{target: diagnostics.CredibleIntervals} from the datasets `load_mcmc` returned (empty when the file has none)"""
    from .diagnostics import CredibleIntervals

    out = {}
    for target in sorted({k.split("/")[1] for k in data if k.startswith("credible/")}):
        f = {k: data[f"credible/{target}/{k}"] for k in ("alpha", "nchains", "nsamples", "lower", "upper")}
        out[target] = CredibleIntervals(float(f["alpha"]), int(f["nchains"]), int(f["nsamples"]), f["lower"], f["upper"])
    return out
