"""Samplers mirroring ``pxmcmc/mcmc.py`` of the reference: ``PxMCMCParams``,
``MYULA``, ``PxMALA``, ``SKROCK`` with the same constructor arguments, ``run``,
``chain_step``, ``logpi``, tracked arrays and traces.

The chain state lives in HBM for the whole run; each iteration is a fixed
sequence of libpxmcmc_b200 kernels.  Two extra keyword-only knobs:

* ``noise="host"`` (default) draws the Gaussian / Laplace / uniform variates from
  numpy's global RNG in exactly the reference's call order, so a seeded run
  reproduces the reference chain (parity mode).  ``noise="device"`` generates
  Philox4x32-10 Gaussians inside the update kernel (throughput mode).
* ``nchains`` runs that many independent chains as one batch (tracked arrays gain
  a leading chain axis when ``nchains > 1``).
* ``summarise=("chain",)`` or ``("chain", "predictions")`` keeps streaming posterior summaries on the device (mean,
  variance, split-R-hat, ESS; see `diagnostics`) instead of, or besides, the tracked arrays: ``sampler.summary`` after
  ``run()``.
* ``credible=("chain",)`` or ``("chain", "predictions")`` keeps the (1 - ``credible_alpha``) credible intervals of
  every element on the device, exactly numpy's quantiles of the samples the tracked arrays would hold, without storing
  them: ``sampler.credible_intervals`` after ``run()``.
"""
import numpy as np
import torch
from scipy.stats import laplace

from . import device as D
from .forward import RingPreds
from .prior import L1, is_library_l1
from .utils import cheb1der, chebyshev1


class PxMCMCParams:
    """Tuning and runtime parameters (pxmcmc/mcmc.py:6-43)."""

    def __init__(
        self,
        lmda=3e-5,
        delta=1e-5,
        s=1,
        mu=1,
        nsamples=int(1e6),
        nburn=int(1e3),
        ngap=int(1e2),
        complex=False,
        verbosity=100,
        track=["logposterior", "L2", "prior", "chain"],
    ):
        self.lmda = lmda
        self.delta = delta
        self.mu = mu
        self.s = s
        self.nsamples = nsamples
        self.nburn = nburn
        self.ngap = ngap
        self.complex = complex
        self.verbosity = verbosity
        self.track = track


def _cplx_lt(a, b):
    """numpy's ordering of complex scalars (real part first, then imaginary),
    which is what `np.log(u) < logalpha` uses when logalpha is complex
    (pxmcmc/mcmc.py:245)."""
    a, b = complex(a), complex(b)
    return (a.real < b.real) or (a.real == b.real and a.imag < b.imag)


class PxMCMC:
    """Common machinery (pxmcmc/mcmc.py:46-140)."""

    def __init__(self, forward, prior, mcmcparams=PxMCMCParams(), *, noise="host", nchains=1, seed=0, stream0=0,
                 spill_dir=None, async_spill=True, summarise=None, credible=None, credible_alpha=0.05):
        """`spill_dir`: directory in which the two large tracked arrays (`chain`, `preds`) live as .npy memory maps
        instead of host RAM (SURVEY.md 8(f)1: 5 000 x 1.22 M samples of config 4 are 49 GB).  `async_spill`: tracked
        samples leave the device through pinned staging buffers on a copy stream while the chain keeps iterating
        (the run loops never wait for a device -> host copy); False restores the synchronous copy.
        `summarise`: None, ("chain",) or ("chain", "predictions"): running moments of every tracked-grid sample are
        kept on the device, independently of `track` (one kernel launch per grid sample and target, no host
        synchronisation, no stored samples); after `run()`, `summary` = {target: diagnostics.Summary} and
        `summary_partials()` the raw partial records (multi-GPU: sharding.gather_summary).
        `credible`: None, ("chain",) or ("chain", "predictions"): the alpha / 2 and 1 - alpha / 2 tails of every
        tracked-grid sample are kept on the device (alpha = `credible_alpha`, one kernel launch per grid sample and
        target, about alpha of the stored chain's memory); after `run()`, `credible_intervals` = {target:
        diagnostics.CredibleIntervals}, bit for bit numpy's quantiles of the samples the tracked arrays would hold."""
        self.forward = forward
        self.prior = prior
        self.spill_dir = spill_dir
        self.async_spill = bool(async_spill)
        for attr in mcmcparams.__dict__.keys():
            setattr(self, attr, getattr(mcmcparams, attr))
        if noise not in ("host", "device"):
            raise ValueError("noise must be 'host' or 'device'")
        self.noise = noise
        self.nchains = int(nchains)
        self.seed = int(seed)
        self.stream0 = int(stream0)  # global index of this sampler's first chain (Philox stream id)
        self._step_counter = 0
        self._summarise = self._check_summarise(summarise)
        self._stats = None
        self._credible = self._check_summarise(credible, "credible")
        alpha = float(credible_alpha)
        if not 0.0 < alpha < 1.0:
            raise ValueError(f"credible_alpha must lie in (0, 1), got {credible_alpha}")
        self._credible_alpha = alpha
        self._cred, self.credible_intervals = None, None
        self._initialise_tracking_arrays()

    # ------------------------------------------------------------------ helpers
    def _native(self):
        return bool(getattr(self.forward, "_pxm_native", False)) and is_library_l1(self.prior)

    def _fused_prox(self):
        """(Tvec, Tscalar) when the prox is a plain soft threshold that the update
        kernel can fuse, else None"""
        if is_library_l1(self.prior) and self.prior.setting == "synthesis":
            return self.prior._T_args()
        return None

    def _ring_mode(self):
        """True when the predictions can be carried as ring-Fourier coefficients (ForwardOperator._ring_fusable): the
        pixel-side ring FFT pair of consecutive iterations cancels"""
        f = getattr(self.forward, "_ring_fusable", None)
        return bool(f is not None and getattr(self.forward, "_pxm_native", False) and f())

    def _initial_preds(self, Xd, P=None):
        """predictions of the state(s) in the form the run loops carry them: `RingPreds` in ring mode, else pixels.
        `P`: the predictions of Xd when known, kept unless they are pixels and the loops carry ring coefficients"""
        if self._ring_mode() and not isinstance(P, RingPreds):
            return self.forward.forward_ring(Xd)
        return D.to_dev_c(self._forward_dev(Xd)) if P is None else P

    @staticmethod
    def _pix(P):
        """pixel-space predictions [nchains, ndata] whatever form they are carried in"""
        return P.pixels() if isinstance(P, RingPreds) else P

    def _state(self, X):
        """[nchains, nparams] complex device tensor from a numpy vector / tensor"""
        x = D.to_dev_c(X)
        return x.unsqueeze(0) if x.dim() == 1 else x

    def _prior_dev(self, Xd):
        if is_library_l1(self.prior):
            return D.reduce_dev(0, Xd, w=self.prior._weights_dev()).real
        vals = [self.prior.prior(D.to_host(Xd[c])) for c in range(Xd.shape[0])]
        return torch.as_tensor(np.real(vals), device=Xd.device)

    def _proxf_dev(self, Xd):
        if is_library_l1(self.prior):
            return D.to_dev_c(self.prior.proxf(Xd))
        return torch.stack([D.to_dev_c(self.prior.proxf(D.to_host(Xd[c]))) for c in range(Xd.shape[0])])

    def _forward_dev(self, Xd, out=None):
        """predictions of the state(s); `out`: buffer the result must end up in (captured graphs: the operator's last
        kernel writes straight into it, see device.output_into)"""
        if getattr(self.forward, "_pxm_native", False):
            if out is None:
                return self.forward.forward(Xd)
            with D.output_into(out):
                r = D.to_dev_c(self.forward.forward(Xd))
            return D.copy_into(out, r.reshape(out.shape))
        r = torch.stack([D.to_dev_c(self.forward.forward(D.to_host(Xd[c]))) for c in range(Xd.shape[0])])
        return r if out is None else D.copy_into(out, r.reshape(out.shape))

    def _gradg_dev(self, Pd):
        if getattr(self.forward, "_pxm_native", False):
            return self.forward.calc_gradg(Pd)
        return torch.stack([D.to_dev_c(self.forward.calc_gradg(D.to_host(Pd[c]))) for c in range(Pd.shape[0])])

    def _logpi_dev(self, Xd, Pd):
        """per-chain (logPi, L2, prior) as host numpy arrays (complex, complex, real)"""
        red = getattr(self.forward, "_pxm_allreduce", None)  # m-sharded operator: partial sums per rank
        if getattr(self.forward, "_diag", None) is not None:
            data_d, ic_d = self.forward._upload()
            L2d = D.reduce_dev(1, Pd, b=data_d, c=ic_d)
            L2 = D.to_host(red(L2d) if red else L2d)
        else:
            L2 = np.array([self._host_L2(D.to_host(Pd[c])) for c in range(Pd.shape[0])])
        prd = self._prior_dev(Xd)
        pr = D.to_host(red(prd) if red else prd)
        return -self.mu * pr - L2, L2, pr

    def _logpi_terms_dev(self, Xd, Pd):
        """(L2, prior) as DEVICE tensors [nchains] (complex, real), or None when the operator has a
        general covariance (host path)"""
        if getattr(self.forward, "_diag", None) is None or not is_library_l1(self.prior):
            return None
        red = getattr(self.forward, "_pxm_allreduce", None)
        data_d, ic_d = self.forward._upload()
        L2d = D.reduce_dev(1, Pd, b=data_d, c=ic_d)
        prd = self._prior_dev(Xd)
        return (red(L2d) if red else L2d), (red(prd) if red else prd)

    def _host_L2(self, preds):
        diff = np.asarray(self.forward.data) - preds
        return np.vdot(diff, self.forward.invcov @ diff)

    # ------------------------------------------------------------------ reference API
    graph_run = True  # run(): replay the iteration as one CUDA graph when it can be recorded (`_graphed`)
    _burn_in_line = False  # run() prints "Burning in..." at the progress steps of the burn-in (the reference's MYULA)
    _pair_engine = None  # MYULA(real_pairs=True): the sampler that iterates on the packed chains

    @property
    def engine(self):
        """the sampler whose `iterate` / `capture` / `iterate_host` act on the device representation of the chains:
        the packed one in `real_pairs` mode, else this sampler itself"""
        return self._pair_engine if self._pair_engine is not None else self

    def _graphed(self):
        """True when run() replays the iteration as one CUDA graph: `graph_run`, Philox noise (host draws cannot be
        recorded) and every operation of the iteration on the device (native operator and prior, not m-sharded).
        Small bandlimits are launch-latency bound: 85 -> 63 us per MYULA iteration at L = 32."""
        eng = self.engine
        return bool(self.graph_run and self.noise == "device" and eng._native()
                    and getattr(eng.forward, "_pxm_allreduce", None) is None)

    def run(self, start_point=None, *, checkpoint=None, checkpoint_every=0, resume=None):
        """the loop of pxmcmc/mcmc.py:150-183 (MYULA) and :308-336 (SKROCK) on the device state `engine` iterates.
        Extensions (keyword-only): `checkpoint` = file written every `checkpoint_every` iterations (and at the end);
        `resume` = such a file: the chain continues exactly as if it had never stopped (same Philox steps / same numpy
        RNG stream, tracked arrays restored).  In `real_pairs` mode samples are unpacked where they are tracked or
        checkpointed (every `ngap`-th iteration), so the tracked arrays are the ordinary ones; the summaries take the
        packed chains."""
        eng = self.engine
        pairs = eng is not self
        i = 0
        j = 0
        self._stats_begin(eng.nchains, pairs=pairs)
        if resume is not None:
            i, j, X, P = self.load_checkpoint(resume)
        else:
            X, P = self._initial_sample(start_point, want_preds=False)
        if pairs:  # the packed engine computes its own predictions
            eng._step_counter = self._step_counter
            X, P = self.pack(X), None
        P = eng._initial_preds(X, P)

        def outer(X, P):
            """state and predictions as the tracked arrays and checkpoints hold them"""
            return (self.unpack(X), self.unpack(eng._pix(P))) if pairs else (X, P)

        graphed = eng.capture(X, P) if self._graphed() else None
        while j < self.nsamples:
            if graphed is not None:
                graphed.step()
                X, P = graphed._state_raw()
            else:
                X, P = eng.iterate(X, P)
            self._step_counter = eng._step_counter
            if self._on_grid(i):
                P_pix = eng._pix(P)
                self._track_dev(j, *outer(X, P_pix))
                self._stats_push(X, P_pix, j)
                j += 1
            if self.verbosity > 0 and (i + 1) % self.verbosity == 0:
                if i >= self.nburn:
                    self._track_flush()
                    self._print_progress(j - 1, np.ravel(self.logPi)[j - 1], L2=np.ravel(self.L2s)[j - 1],
                                         prior=np.ravel(self.priors)[j - 1])
                elif self._burn_in_line:
                    print("Burning in...")
            i += 1
            if checkpoint is not None and checkpoint_every and i % checkpoint_every == 0:
                self.save_checkpoint(checkpoint, i, j, *outer(X, P))
        if checkpoint is not None:
            self.save_checkpoint(checkpoint, i, j, *outer(X, P))
        self._track_flush()
        self._stats_end()
        self._final_state = outer(X, eng._pix(P))
        if graphed is not None:
            graphed.release()
        print("\nDONE")

    def capture(self, X, P=None, iterations=1):
        """Record `iterations` passes of `iterate` as ONE CUDA graph on private copies of the state and return a
        `GraphedChain`: `.step()` replays it (a single launch instead of ~10-40 kernel launches per MYULA iteration and
        ~14 per stage of a SKROCK step: single-chain runs are launch-latency bound, SURVEY.md 7.2), `.state()` returns the
        current (X, preds).  `P`: the predictions of X (computed here when None).  Needs `noise="device"` (the Philox
        step then lives in device memory and is advanced inside the graph; the noise stream is the same as without the
        graph)."""
        if self.noise != "device":
            raise ValueError("capture() needs noise='device' (host RNG draws cannot be recorded)")
        return GraphedChain(self, X, P, iterations)

    def logpi(self, X, preds):
        """log posterior, L2 misfit and prior of a model (pxmcmc/mcmc.py:71-82):
        L2 = vdot(d, invcov d) with d = data - preds, logPi = -mu*prior - L2."""
        lp, l2, pr = self._logpi_dev(self._state(X), self._state(preds))
        return lp[0], l2[0], pr[0]

    def _gradg_at(self, Xd, Pd=None):
        """gradg of the predictions of Xd (computed here unless `Pd` is given), as a device tensor"""
        if Pd is None and self._ring_mode():
            return self.forward.gradg_from_ring(self.forward.forward_ring(Xd))
        if Pd is None:
            Pd = self._forward_dev(Xd)
        return D.to_dev_c(self._gradg_dev(self._pix(Pd)))

    def _gradlogpi_dev(self, Xd, Pd=None):
        gradg = self._gradg_at(Xd, Pd)
        fused = self._fused_prox()
        if fused is not None:
            return D.gradlogpi_dev(Xd, None, fused[0], fused[1], gradg, self.lmda)
        return D.gradlogpi_dev(Xd, self._proxf_dev(Xd), None, 0.0, gradg, self.lmda)

    def _gradlogpi(self, X, preds=None):
        """-(X - prox(X))/lmda - gradg(forward(X)) (pxmcmc/mcmc.py:84-89)"""
        out = self._gradlogpi_dev(self._state(X), None if preds is None else self._state(preds))
        return out if D.is_dev(X) else D.to_host(out[0])

    def _print_progress(self, i, logpi, **kwargs):
        print(
            f"{i+1:,}/{self.nsamples:,} - logposterior: {logpi:.8e} - "
            + " - ".join([f"{k}: {kwargs[k]:.8e}" for k in kwargs]),
        )

    def _initial_sample(self, initial_sample=None, want_preds=True):
        """Laplace draw (or the user's 1-D start point), and its predictions
        (pxmcmc/mcmc.py:97-111).  Returns device tensors [nchains, .]."""
        n = self.forward.nparams
        if initial_sample is None:
            X = laplace.rvs(size=n * self.nchains)
            if self.complex:
                X = X + laplace.rvs(size=n * self.nchains) * 1j
            X = X.reshape(self.nchains, n)
        else:
            if D.is_dev(initial_sample):
                X = initial_sample
                if X.shape[-1] != n:
                    raise ValueError("Inital sample given has incorrect size")
            else:
                if not isinstance(initial_sample, np.ndarray) or np.ndim(initial_sample) not in (1, 2):
                    raise TypeError("Expected a 1D numpy array as an initial sample")
                if np.ndim(initial_sample) == 2 and self.nchains == 1:
                    raise TypeError("Expected a 1D numpy array as an initial sample")
                if initial_sample.shape[-1] != n:
                    raise ValueError("Inital sample given has incorrect size")
                X = initial_sample
                if np.ndim(X) == 1 and self.nchains > 1:
                    X = np.tile(X, (self.nchains, 1))
        Xd = self._state(X)
        return Xd, (D.to_dev_c(self._forward_dev(Xd)) if want_preds else None)

    # ------------------------------------------------------------------ MAP estimate (FISTA), step-size bound
    _FISTA_BLOCK = 50  # iterations between two convergence reads (one CUDA graph replay when graphed)

    # p = delta * Lip(grad log pi) up to which one step is stable (the samplers that have such a bound override it)
    stability_limit = float("nan")

    def max_stable_delta(self):
        """stability_limit / (L_f + 1 / lmda): the largest step size delta for which one step of the sampler is stable
        (its deterministic factor on a quadratic stays within [-1, 1]), with L_f = `forward.lipschitz()` the Lipschitz
        constant of gradg and 1 / lmda that of the Moreau-Yosida term.  A stability bound, not an accuracy
        recommendation: the chain's bias grows with delta below it too.  Synthesis setting, library L1 prior,
        real positive inverse covariance (the refusals of `map_estimate`).  NaN when the sampler has no stability
        limit (SKROCK's reference scheme)."""
        if np.isnan(self.stability_limit):
            return float("nan")
        self._check_map_problem("max_stable_delta")
        return self.stability_limit / (self.forward.lipschitz() + 1.0 / self.lmda)

    def _check_map_problem(self, what):
        """raise unless the drift -(x - prox x)/lmda - gradg(x) is the Moreau-Yosida gradient flow of the real objective
        F(x) = 1/2 (Phi Psi x - d)^dagger IC (Phi Psi x - d) + mu sum_i w_i |x_i| (see `map_estimate`)"""
        if self.forward.setting != "synthesis" or getattr(self.prior, "setting", None) != "synthesis":
            raise NotImplementedError(
                f"{what}: the analysis setting is not supported (the reference's analysis prox X + Psi(soft(Psi^dagger X) "
                "- Psi^dagger X) is not the prox of mu ||w Psi^dagger x||_1)")
        if not is_library_l1(self.prior):
            raise NotImplementedError(f"{what}: a user-overridden prox / prior is not supported (the library's L1 "
                                      "priors only: the prox must be the soft threshold)")
        if getattr(self.forward, "_diag", None) is None:
            raise NotImplementedError(f"{what}: a full covariance matrix is not supported (diagonal covariances only)")
        if getattr(self.forward, "_pxm_allreduce", None) is not None:
            raise NotImplementedError(f"{what}: m-sharded operators are not supported")
        why = self.forward._real_positive_ic()
        if why is not None:
            raise ValueError(f"{what}: {why}")

    def _map_objective(self, Xd):
        """F of every chain of Xd [nchains, n] as a float64 device tensor: 1/2 L2 + mu prior (pxm_reduce kinds 1, 0).
        The tracked logPi = -mu prior - L2 has no 1/2 (as in the reference), so F is not -logPi."""
        L2, pr = self._logpi_terms_dev(Xd, D.to_dev_c(self._forward_dev(Xd)))
        return 0.5 * L2.real + self.mu * pr

    def map_estimate(self, start_point=None, *, tol=1e-8, maxiter=100_000):
        """MAP estimate of the synthesis-setting posterior by FISTA (Beck & Teboulle 2009) on the device: the minimiser
        of F(x) = 1/2 (Phi Psi x - d)^dagger IC (Phi Psi x - d) + mu sum_i w_i |x_i| (|.| the complex modulus, as the
        soft threshold), whose Moreau-Yosida gradient flow is the samplers' drift -(x - prox(x))/lmda - gradg(x) when
        the prior's threshold is T = lmda mu w (the library's L1 priors, is_library_l1).  F carries the 1/2 the tracked
        log posterior (-mu prior - L2, as in the reference) does not have: F is not -logPi.

        Step t = 1 / L_f (`forward.lipschitz()`), threshold (t / lmda) T.  `start_point`: None (a Laplace draw) or a
        start point, with the conventions of `run`; every chain is solved independently.  Stops when the largest
        relative change |x_{k+1} - x_k| / |x_{k+1}| over the chains is below `tol`, read once every block of
        iterations (one small device -> host copy), or after `maxiter` iterations.  A block is one CUDA graph when the
        operator and prior are native, else it runs eagerly; both give the same iterates bit for bit.  With
        `real_pairs=True` the problem is solved on the operator given to the sampler.

        Returns (x, info): x complex [n] (one chain) or [nchains, n], a valid `run(start_point=x)`; info = {"F":
        objective per chain at x, "iterations", "converged", "relative_change": [blocks, nchains] at the end of every
        block, "F_history": [blocks, nchains], "lipschitz": L_f, "step": t}.

        Raises NotImplementedError in the analysis setting, for a user-overridden prox or prior, a full covariance
        matrix or an m-sharded operator, and ValueError when the inverse covariance is not real and positive (the
        reference's rule var (1 + i) / sqrt 2 for a real sigma with complex data: pass sigma as a complex array)."""
        self._check_map_problem("map_estimate")
        Lf = self.forward.lipschitz()
        t = 1.0 / Lf
        Tv, Ts = self._fused_prox()
        X, _ = self._initial_sample(start_point, want_preds=False)
        X = X.clone()
        Y = X.clone()
        nch = X.shape[0]
        K = self._FISTA_BLOCK
        state = torch.tensor([0.0, 1.0], dtype=D.FDT, device=X.device)
        hist = torch.zeros((K, nch, 2), dtype=D.FDT, device=X.device)

        def iteration(x, y, st, h):
            D.fista_update_dev(y, self._gradg_at(y), x, Tv, Ts, t / self.lmda, t, st, h, out=(x, y))

        def warm_up():  # on copies: the state of the solve is not touched
            xw, yw, sw, hw = X.clone(), Y.clone(), state.clone(), hist.clone()
            for _ in range(2):
                iteration(xw, yw, sw, hw)

        def block():
            for _ in range(K):
                iteration(X, Y, state, hist)

        graph = None
        if self._native() and maxiter >= K:
            _warm_up(warm_up)
            graph = _record_graph(block)
        its, converged, rel, Fh = 0, False, [], []
        while its < maxiter and not converged:
            k = min(K, maxiter - its)
            if graph is not None and k == K:
                graph.replay()
            else:
                for _ in range(k):
                    iteration(X, Y, state, hist)
            its += k
            F = self._map_objective(X)
            v = torch.cat([hist[(its - 1) % K].reshape(-1), F]).cpu().numpy()
            dx2, x2 = v[0:2 * nch:2], v[1:2 * nch:2]
            r = np.sqrt(dx2) / np.maximum(np.sqrt(x2), np.finfo(float).tiny)
            rel.append(r)
            Fh.append(v[2 * nch:])
            converged = bool(np.max(r) < tol)
        out = D.to_host(X)
        if self.nchains == 1:
            out = out[0]
        info = {"F": Fh[-1] if nch > 1 else float(Fh[-1][0]), "iterations": its, "converged": converged,
                "relative_change": np.array(rel), "F_history": np.array(Fh), "lipschitz": Lf, "step": t}
        return out, info

    def _initialise_tracking_arrays(self):
        """pxmcmc/mcmc.py:113-128 (leading chain axis only when nchains > 1)"""
        lead = (self.nchains,) if self.nchains > 1 else ()
        if "logposterior" in self.track:
            self.logPi = np.zeros(lead + (self.nsamples,))
        def big(name, shape, dtype):
            if self.spill_dir is None:
                return np.zeros(shape, dtype=dtype)
            import os

            os.makedirs(self.spill_dir, exist_ok=True)
            return np.lib.format.open_memmap(os.path.join(self.spill_dir, name + ".npy"), mode="w+", dtype=dtype, shape=shape)

        if "predictions" in self.track:
            self.preds = big("predictions", lead + (self.nsamples, len(self.forward.data)), float)
        if "chain" in self.track:
            self.chain = big("chain", lead + (self.nsamples, self.forward.nparams), complex if self.complex else float)
        if "L2" in self.track:
            self.L2s = np.zeros(lead + (self.nsamples,), dtype=float)
        if "prior" in self.track:
            self.priors = np.zeros(lead + (self.nsamples,), dtype=float)

    def _put(self, arr, j, val, c=slice(None)):
        """store sample j of chain(s) `c` (all by default) in a tracked array; complex values are truncated to their
        real part exactly as numpy does when the reference assigns them into float arrays (pxmcmc/mcmc.py:130-140)"""
        val = np.asarray(val)
        if not np.iscomplexobj(arr):
            val = val.real
        if self.nchains > 1:
            arr[c, j] = val
        else:
            arr[j] = val[0] if val.ndim and val.shape[0] == 1 else val

    def _tracking(self, j, X_curr, curr_preds, logPi, L2, prior):
        """store sample j of every chain (pxmcmc/mcmc.py:130-140)"""
        if hasattr(self, "logPi"):
            self._put(self.logPi, j, logPi)
        if hasattr(self, "L2s"):
            self._put(self.L2s, j, L2)
        if hasattr(self, "priors"):
            self._put(self.priors, j, prior)
        if hasattr(self, "preds"):
            self._put(self.preds, j, D.to_host(curr_preds) if D.is_dev(curr_preds) else curr_preds)
        if hasattr(self, "chain"):
            self._put(self.chain, j, D.to_host(X_curr) if D.is_dev(X_curr) else X_curr)

    def _track_dev(self, j, X_curr, curr_preds):
        """sample j of a device-resident chain: log posterior terms and the tracked vectors.  With `async_spill` nothing
        here waits for the device: the reductions stay device tensors, state and predictions are snapshotted on the
        compute stream and leave through `_Spill`; the host arrays are filled when the slot is reused, on `flush`, or
        before anything reads them (progress lines, checkpoints, the end of `run`)."""
        curr_preds = self._pix(curr_preds)
        terms = self._logpi_terms_dev(X_curr, curr_preds) if self.async_spill else None
        if terms is None:
            logPi, L2, prior = self._logpi_dev(X_curr, curr_preds)
            self._tracking(j, X_curr, curr_preds, logPi, L2, prior)
            return
        if getattr(self, "_spill", None) is None:
            self._spill = _Spill(self)
        self._spill.push(j, X_curr, curr_preds, terms[0], terms[1])

    def _track_flush(self):
        if getattr(self, "_spill", None) is not None:
            self._spill.flush()

    # ------------------------------------------------------------------ checkpoint / resume
    _TRACKED = ("logPi", "L2s", "priors", "preds", "chain")

    def _save_ckpt(self, path, **fields):
        """One .npz (written to a temporary name, then renamed) with `fields` plus everything every sampler needs to
        continue exactly where it stands: the Philox step, the step size, numpy's global RNG state (host-noise mode)
        and the tracked arrays filled so far."""
        import os

        self._track_flush()
        d = dict(fields)
        d.update(step_counter=self._step_counter, nchains=self.nchains, noise=self.noise, delta=self.delta,
                 sampler=type(self).__name__)
        for name in self._TRACKED:
            if hasattr(self, name):
                d["track_" + name] = getattr(self, name)
        if self._stats is not None:
            d.update({"stats_" + k: v for k, v in self._stats.state().items()})
        if self._cred is not None:
            d.update({"cred_" + k: v for k, v in self._cred.state().items()})
        kind, keys, pos, has_gauss, cached = np.random.get_state()
        d.update(rng_keys=keys, rng_pos=pos, rng_has_gauss=has_gauss, rng_cached=cached)
        tmp = path + ".tmp.npz"
        np.savez(tmp, **d)
        os.replace(tmp, path if path.endswith(".npz") else path + ".npz")

    def _load_ckpt(self, path):
        """-> dict of the saved fields; restores the tracked arrays, the Philox step, the step size and numpy's RNG state"""
        with np.load(path if path.endswith(".npz") else path + ".npz", allow_pickle=False) as f:
            if int(f["nchains"]) != self.nchains or str(f["noise"]) != self.noise:
                raise ValueError("checkpoint was written by a sampler with another chain count / noise mode")
            if "sampler" in f.files and str(f["sampler"]) != type(self).__name__:
                raise ValueError(f"checkpoint was written by {f['sampler']}, not {type(self).__name__}")
            for name in self._TRACKED:
                if "track_" + name in f.files and hasattr(self, name):
                    arr = f["track_" + name]
                    if arr.shape != getattr(self, name).shape:
                        raise ValueError(f"checkpoint array {name} has shape {arr.shape}, expected {getattr(self, name).shape}")
                    getattr(self, name)[...] = arr
            if self._stats is not None:
                missing = [k for k in self._stats.acc if "stats_" + k not in f.files]
                if missing:
                    raise ValueError(f"checkpoint carries no summary accumulators for {missing}: it was written by a "
                                     "sampler without summarise=...")
                self._stats.load({k: f["stats_" + k] for k in self._stats.acc})
            if self._cred is not None:
                keys = list(self._cred.heaps) + ["count"]
                missing = [k for k in keys if "cred_" + k not in f.files]
                if missing:
                    raise ValueError(f"checkpoint carries no credible-interval heaps for {missing}: it was written by "
                                     "a sampler without credible=...")
                self._cred.load({k: f["cred_" + k] for k in keys})
            self._step_counter = int(f["step_counter"])
            self.delta = float(f["delta"])
            np.random.set_state(("MT19937", f["rng_keys"], int(f["rng_pos"]), int(f["rng_has_gauss"]), float(f["rng_cached"])))
            return {k: f[k] for k in f.files if not k.startswith(("track_", "rng_", "stats_", "cred_"))}

    def save_checkpoint(self, path, i, j, X_curr, curr_preds):
        """Everything `run(resume=path)` needs to continue the chain exactly where it stands after iteration
        i - 1: state and predictions, loop counters, and the common fields of `_save_ckpt`."""
        extra = {}
        if isinstance(curr_preds, RingPreds):  # the ring coefficients themselves: a resumed chain continues bit for bit
            extra["P_ring"] = D.to_host(curr_preds.t)
            extra["P_kind"] = curr_preds.kind
        self._save_ckpt(path, i=i, j=j, X=D.to_host(X_curr), P=D.to_host(self._pix(curr_preds)), **extra)

    def load_checkpoint(self, path):
        """-> (i, j, X, preds) as device tensors"""
        f = self._load_ckpt(path)
        X = self._state(f["X"])
        if "P_ring" in f and self._ring_mode() and str(f["P_kind"]) == self.forward._ring_kind():
            P = RingPreds(torch.from_numpy(np.ascontiguousarray(f["P_ring"])).to(X.device), self.forward, X.shape[0],
                          str(f["P_kind"]))
        else:
            P = self._state(f["P"])
        return int(f["i"]), int(f["j"]), X, P

    def _on_grid(self, i):
        return i >= self.nburn and (self.ngap == 0 or (i - self.nburn) % self.ngap == 0)

    def _host_noise(self, n):
        """Gaussian draw(s) in the reference's order: real part, then imaginary if `complex`"""
        w_re = D.to_dev_f(np.random.randn(n * self.nchains))
        w_im = D.to_dev_f(np.random.randn(n * self.nchains)) if self.complex else None
        return w_re, w_im

    # ------------------------------------------------------------------ streaming posterior summaries
    def _check_summarise(self, summarise, option="summarise"):
        if summarise is None:
            return ()
        if isinstance(summarise, str):
            summarise = (summarise,)
        t = tuple(summarise)
        if not t or len(set(t)) != len(t) or any(k not in ("chain", "predictions") for k in t):
            raise ValueError(f'{option} must be None, ("chain",) or ("chain", "predictions")')
        if getattr(self.forward, "_pxm_allreduce", None) is not None:
            raise NotImplementedError(f"{option}: streaming {'summaries' if option == 'summarise' else 'intervals'} of "
                                      "m-sharded single-chain runs are not implemented (each rank holds only part of "
                                      "every sample)")
        return t

    def _stats_begin(self, nchains_dev=None, pairs=False):
        """fresh accumulators at the start of run() (nsamples fixes the half-chain and batch boundaries); modes as in
        pxm_stats_accumulate: the chain is complex (re + im) only with `complex`, predictions are real parts"""
        from .diagnostics import StreamingCredible, StreamingSummary

        self._stats, self.summary = None, None
        self._cred, self.credible_intervals = None, None
        nch = self.nchains if nchains_dev is None else nchains_dev

        def layout(targets):
            lay = {}
            if "chain" in targets:
                lay["chain"] = (self.forward.nparams, nch, 2 if pairs else (1 if self.complex else 0))
            if "predictions" in targets:
                lay["predictions"] = (len(self.forward.data), nch, 2 if pairs else 0)
            return lay

        if self._summarise:
            self._stats = StreamingSummary(layout(self._summarise), self.nsamples)
        if self._credible:  # the heaps are sized for the run's pooled sample count
            self._cred = StreamingCredible(layout(self._credible), self.nsamples, self._credible_alpha)

    def _stats_push(self, X, P, j=0, d_j=None, nactive=None):
        """push tracked-grid sample j (per chain: d_j; `nactive` chains take one) of the state X and the PIXEL
        predictions P (may be None when predictions are neither summarised nor bounded)"""
        if self._stats is not None:
            if "chain" in self._stats.acc:
                self._stats.push("chain", X, j, d_j)
            if "predictions" in self._stats.acc:
                self._stats.push("predictions", P, j, d_j)
        if self._cred is not None:
            self._cred.push({"chain": X, "predictions": P}, d_j, nactive)

    def _stats_end(self):
        if self._cred is not None:
            self.credible_intervals = self._cred.intervals()
        if self._stats is None:
            return
        from .diagnostics import finalize

        self._partials = self._stats.partials()
        self.summary = {k: finalize([p]) for k, p in self._partials.items()}

    def summary_partials(self):
        """{target: partial record dict} of the last run (combine several with diagnostics.finalize or
        sharding.gather_summary)"""
        if getattr(self, "_partials", None) is None:
            raise RuntimeError("no summary: construct the sampler with summarise=... and call run()")
        return self._partials


class _Spill:
    """Non-blocking device -> host spill of tracked samples (SURVEY.md 8(f)1).  Two slots; a slot holds a device
    snapshot of (X, preds, L2, prior) taken on the compute stream -- the chain overwrites its state in place on the
    next iteration -- and pinned host buffers filled by a copy stream.  The host arrays are written when a slot is
    reused (two samples later: the copy has long finished) or on `flush`."""

    def __init__(self, sampler):
        self.s = sampler
        self.stream = torch.cuda.Stream()
        self.slots = [None, None]
        self.want_chain, self.want_preds = hasattr(sampler, "chain"), hasattr(sampler, "preds")

    def _alloc(self, X, P, L2):
        def pair(t):
            return torch.empty_like(t), torch.empty(t.shape, dtype=t.dtype).pin_memory()

        d = {"L2": pair(L2), "prior": pair(L2.real.contiguous()), "done": torch.cuda.Event(), "j": None}
        if self.want_chain:
            d["X"] = pair(X)
        if self.want_preds:
            d["P"] = pair(P)
        return d

    def push(self, j, X, P, L2, prior):
        k = j & 1
        if self.slots[k] is None:
            self.slots[k] = self._alloc(X, P, L2)
        sl = self.slots[k]
        self._write(sl)
        cur = torch.cuda.current_stream()
        items = [("L2", L2), ("prior", prior)] + ([("X", X)] if self.want_chain else []) + ([("P", P)] if self.want_preds else [])
        for name, t in items:
            sl[name][0].copy_(t.reshape(sl[name][0].shape))  # device snapshot, ordered after the iteration
        ready = torch.cuda.Event()
        ready.record(cur)
        self.stream.wait_event(ready)
        with torch.cuda.stream(self.stream):
            for name, _ in items:
                sl[name][1].copy_(sl[name][0], non_blocking=True)
            sl["done"].record(self.stream)
        # (the compute stream never waits for the spill: the next snapshot into this slot is two samples away and
        # `_write` has synchronised on `done` by then)
        sl["j"] = j

    def _write(self, sl):
        if sl is None or sl["j"] is None:
            return
        sl["done"].synchronize()
        s, j = self.s, sl["j"]
        L2 = sl["L2"][1].numpy()
        pr = sl["prior"][1].numpy()
        logPi = -s.mu * pr - L2
        X = sl["X"][1].numpy() if self.want_chain else None
        P = sl["P"][1].numpy() if self.want_preds else None
        s._tracking(j, X, P, logPi, L2, pr)
        sl["j"] = None

    def flush(self):
        for sl in sorted([x for x in self.slots if x is not None and x["j"] is not None], key=lambda x: x["j"]):
            self._write(sl)


class MYULA(PxMCMC):
    """Moreau-Yosida unadjusted Langevin algorithm (pxmcmc/mcmc.py:143-201)."""

    _burn_in_line = True
    # one step on a quadratic multiplies the deviation from the mode by 1 - p, p = delta * Lip(grad log pi): within
    # [-1, 1] for p <= 2
    stability_limit = 2.0

    def __init__(self, forward, prox, mcmcparams=PxMCMCParams(), *, real_pairs=False, **kw):
        """`real_pairs=True` (extension; an even number of chains, real data, real noise level, `complex=False`, the
        library's synthesis-setting L1 prior): real chain 2k travels in the real and chain 2k+1 in the imaginary part
        of ONE complex chain on the device.  Every linear operator of the synthesis path is complex-linear and maps
        real fields to real fields, so the two parts never mix: the transforms of two chains for the price of one (the
        reference carries the same real chain as a complex array with a zero imaginary part).  `run()`, the tracked
        arrays, checkpoints and start points stay in the ordinary [nchains, n] form; `engine` is the sampler that
        iterates on the packed state, `pack` / `unpack` convert.  Chain c draws the Philox stream it would draw
        unpacked."""
        super().__init__(forward, prox, mcmcparams, **kw)
        self.real_pairs = bool(real_pairs)
        self._pair_engine = self._make_pair_engine() if self.real_pairs else None

    # ------------------------------------------------------------------ real chain pairs
    def _make_pair_engine(self):
        import copy

        if type(self) is not MYULA:
            raise ValueError("real_pairs is a MYULA mode")
        if self.nchains < 2 or self.nchains % 2:
            raise ValueError("real_pairs needs an even number of chains")
        if self.complex:
            raise ValueError("real_pairs: the noise must be real (complex=False)")
        if self._fused_prox() is None or not hasattr(self.forward, "paired"):
            raise ValueError("real_pairs needs the library's forward operator and synthesis-setting L1 prior")
        eng = copy.copy(self)
        eng.forward = self.forward.paired()  # ValueError with the reason when the operator cannot be paired
        eng.nchains = self.nchains // 2
        eng.real_pairs, eng._pair_engine, eng._is_pair_engine = False, None, True
        eng._spill = None
        return eng

    @staticmethod
    def pack(X):
        """[2k, n] real-valued chains -> [k, n] complex: chain 2c + i chain (2c+1)"""
        x = D.to_dev_c(X)
        if x.dim() != 2 or x.shape[0] % 2:
            raise ValueError("pack: an even number of chains [nchains, n]")
        if bool(torch.any(x.imag != 0)):
            raise ValueError("pack: the chains must be real-valued")
        return torch.complex(x[0::2].real, x[1::2].real).contiguous()

    @staticmethod
    def unpack(Xp):
        """[k, n] packed chains -> [2k, n] complex tensors with zero imaginary parts"""
        xp = D.to_dev_c(Xp)
        xp = xp.unsqueeze(0) if xp.dim() == 1 else xp
        out = torch.zeros((2 * xp.shape[0], xp.shape[1]), dtype=xp.dtype, device=xp.device)
        out[0::2] = xp.real
        out[1::2] = xp.imag
        return out

    def _propose_dev(self, Xd, proxd, gradgd, out=None):
        """X' = (1-d/l) X + (d/l) prox - d gradg + sqrt(2d) w, one fused kernel;
        proxd None -> the soft threshold is evaluated inside the kernel; `out` (may be Xd itself) receives X'"""
        n = self.forward.nparams
        if proxd is None:
            Tv, Ts = self._fused_prox()
        else:
            Tv, Ts = None, 0.0
        pair = getattr(self, "_is_pair_engine", False)  # packed real chain pairs: kernel modes 4 (Philox) / 5 (injected)
        if pair and proxd is not None:
            raise ValueError("real_pairs: the prox is the library's fused soft threshold")
        mode = 4 if pair else (3 if self.complex else 2)
        if self.noise == "host":
            if pair:  # the draw of the unpacked sampler (one randn over all real chains, chain-major), then packed
                w = np.random.randn(2 * self.nchains, n)
                w_re, w_im = D.to_dev_f(np.ascontiguousarray(w[0::2])), D.to_dev_f(np.ascontiguousarray(w[1::2]))
            else:
                w_re, w_im = self._host_noise(n)
            out = D.myula_update_dev(Xd, proxd, gradgd, Tv, Ts, self.delta, self.lmda, w_re=w_re, w_im=w_im,
                                     noise_mode=5 if pair else 1, out=out)
        elif getattr(self, "_dstep", None) is not None:
            # graph mode: the step lives on the device and is advanced by the captured graph itself
            out = D.myula_update_dev(Xd, proxd, gradgd, Tv, Ts, self.delta, self.lmda,
                                     noise_mode=mode, seed=self.seed, stream0=self.stream0,
                                     dstep=self._dstep, out=out)
        else:
            # chain-group calls of one iteration (iterate_host) share a step; their Philox streams are
            # offset so that chain c always uses stream stream0 + c, whatever the grouping
            off = getattr(self, "_group_offset", None)
            if off is None:
                self._step_counter += 1
            out = D.myula_update_dev(Xd, proxd, gradgd, Tv, Ts, self.delta, self.lmda,
                                     noise_mode=mode, seed=self.seed, step=self._step_counter,
                                     stream0=self.stream0 + (2 if pair else 1) * (off or 0), out=out)
        return out

    def iterate(self, X_curr, curr_preds, out=None):
        """One pass of the loop body (pxmcmc/mcmc.py:158-164) on device tensors
        [nchains, .]: gradg -> prox -> proposal -> new predictions.  `out = (X_buf, P_buf)`: where the new state and
        predictions are written; the input buffers themselves are allowed (the update is elementwise and the old
        predictions are consumed before the new ones are produced), which is how captured graphs advance in place."""
        if isinstance(curr_preds, RingPreds):
            # ring mode: the gradient starts from, and the new predictions stop at, the ring coefficients of the image
            gradg = self.forward.gradg_from_ring(curr_preds)
            proxf = None if self._fused_prox() is not None else self._proxf_dev(X_curr)
            X_new = self._propose_dev(X_curr, proxf, gradg, out=None if out is None else out[0])
            return X_new, self.forward.forward_ring(X_new, out=None if out is None else out[1])
        gradg = D.to_dev_c(self._gradg_dev(curr_preds))
        proxf = None if self._fused_prox() is not None else self._proxf_dev(X_curr)
        if out is None:
            X_new = self._propose_dev(X_curr, proxf, gradg)
            return X_new, D.to_dev_c(self._forward_dev(X_new))
        X_new = self._propose_dev(X_curr, proxf, gradg, out=out[0])
        return X_new, self._forward_dev(X_new, out=out[1])

    def iterate_host(self, X_host, preds_host=None, X_out=None, preds_out=None, groups=None):
        """The same iteration through HOST buffers (pinned torch CPU tensors or numpy
        arrays [nchains, .]): copies the state in, runs the kernels, copies the new
        state and predictions back.  This is the end-to-end path bench.py times.

        `preds_host=None`: state in, state out -- the predictions of the incoming state are recomputed on the device
        (in the form the run loops carry them, see `_initial_preds`) instead of travelling over PCIe, and the new
        predictions are returned only when `preds_out` is given; `chain_step` of the reference likewise maps a state to
        a state (pxmcmc/mcmc.py:185-201).

        With several chains the batch is cut into `groups` chain groups (a count, or a list of group
        sizes) that flow through a
        three-stage pipeline on three CUDA streams -- host->device copy of group g+1, kernels of
        group g, device->host copy of group g-1 -- so that both PCIe directions and the SMs work at
        the same time (the transfers, not the kernels, bound this path).  Results do not depend on
        the grouping: chains are independent and chain c always draws Philox stream stream0 + c.

        Returns (X_out, preds_out), or X_out alone when predictions neither come in nor go out.  Outputs not given are
        pinned tensors allocated here; with predictions in, no outputs and one chain group they are numpy arrays."""
        if self._summarise:
            raise NotImplementedError("summarise: iterate_host has no tracking grid (run() does); use a sampler "
                                      "without summarise=...")
        if self._credible:
            raise NotImplementedError("credible: iterate_host has no tracking grid (run() does); use a sampler "
                                      "without credible=...")
        dv = D.dev()
        as_in = lambda a: a if D.is_dev(a) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.complex128))
        as_out = lambda a: torch.from_numpy(a) if isinstance(a, np.ndarray) else a  # numpy outputs are filled in place
        xh = as_in(X_host)
        xh = xh.unsqueeze(0) if xh.dim() == 1 else xh
        ph = None if preds_host is None else as_in(preds_host).reshape(xh.shape[0], -1)
        nch = xh.shape[0]
        sizes = self._group_sizes(nch, groups)
        as_numpy = ph is not None and X_out is None and len(sizes) == 1
        if X_out is None:
            X_out = torch.empty(xh.shape, dtype=xh.dtype, pin_memory=True)
            if ph is not None:
                preds_out = torch.empty(ph.shape, dtype=ph.dtype, pin_memory=True)
        xo = as_out(X_out).reshape(xh.shape)
        po = None if preds_out is None else as_out(preds_out).reshape(nch, -1)
        st = getattr(self, "_pipe_streams", None)
        if st is None:
            st = self._pipe_streams = (torch.cuda.Stream(), torch.cuda.Stream())
        s_in, s_out = st
        s_cmp = torch.cuda.current_stream()
        s_in.wait_stream(s_cmp)
        starts = [sum(sizes[:g]) for g in range(len(sizes))]
        if self.noise == "device":  # one Philox step for the whole batch, every group at its chains' streams
            self._step_counter += 1
        staged = []
        for g in range(len(sizes)):  # all uploads are queued first: the copy engine never waits for the host
            with torch.cuda.stream(s_in):
                sl = slice(starts[g], starts[g] + sizes[g])
                Xd = xh[sl].to(dv, non_blocking=True)
                Pd = None if ph is None else ph[sl].to(dv, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(s_in)
            staged.append((sl, Xd, Pd, ev))
        try:
            for g, (sl, Xd, Pd, ev) in enumerate(staged):
                s_cmp.wait_event(ev)
                Xd.record_stream(s_cmp)
                if Pd is None:
                    Pd = self._initial_preds(Xd)
                else:
                    Pd.record_stream(s_cmp)
                self._group_offset = starts[g]
                Xn, Pn = self.iterate(Xd, Pd)
                if po is not None:
                    Pn = self._pix(Pn)
                done = torch.cuda.Event()
                done.record(s_cmp)
                s_out.wait_event(done)
                with torch.cuda.stream(s_out):
                    Xn.record_stream(s_out)
                    xo[sl].copy_(Xn, non_blocking=True)
                    if po is not None:
                        Pn.record_stream(s_out)
                        po[sl].copy_(Pn, non_blocking=True)
        finally:
            self._group_offset = None
        s_out.synchronize()
        if as_numpy:
            return X_out.numpy(), preds_out.numpy()
        return X_out if preds_out is None else (X_out, preds_out)

    def _group_sizes(self, nch, groups):
        """chain-group sizes of `iterate_host` from `groups` (None: 8 or 4 groups for wide batches, else 1; a count,
        1 when it does not divide the batch; a list of sizes); one group with host noise (one numpy draw per call)"""
        if groups is None:
            groups = 8 if (nch >= 64 and nch % 8 == 0) else (4 if (nch >= 16 and nch % 4 == 0) else 1)
        if isinstance(groups, int):
            if nch % groups or self.noise != "device" and groups > 1:
                groups = 1
            return [nch // groups] * groups
        sizes = [int(g) for g in groups]
        if sum(sizes) != nch or min(sizes) < 1:
            raise ValueError("group sizes must be positive and add up to the number of chains")
        return sizes if self.noise == "device" else [nch]

    def chain_step(self, X, proxf, gradg):
        """One proposal from (X, prox(X), gradg) (pxmcmc/mcmc.py:185-201)."""
        out = self._propose_dev(self._state(X), self._state(proxf), self._state(gradg))
        return out if D.is_dev(X) else D.to_host(out[0] if np.ndim(X) == 1 else out)


def _warm_up(body):
    """run body() on a side stream and wait for it: tables, lazy uploads, kernel attributes and allocator pools are
    ready before a CUDA graph capture, which must not create them"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()


def _record_graph(body):
    """body() recorded as one CUDA graph on a side stream (the capture executes nothing); the current stream waits
    for the side stream"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        body()
    torch.cuda.current_stream().wait_stream(side)
    return graph


class GraphedChain:
    """`iterations` passes of a sampler's `iterate` as one CUDA graph (see `PxMCMC.capture`).  The chain advances IN
    PLACE: the update kernel (SKROCK: the last stage) writes X and the operator's last kernel writes P, so the graph
    holds no copy-back and no ATen kernel.

    Philox step: the graph reads and advances the device counter `dstep`, which this object keeps alive.
    `sampler._dstep` points to it only while the graph is warmed up and recorded, so eager calls on the sampler draw
    the host counter `sampler._step_counter`, and `step()` advances that counter with the graph."""

    def __init__(self, sampler, X, P=None, iterations=1):
        self.sampler, self.iterations = sampler, int(iterations)
        self.X = sampler._state(X).clone()
        if P is not None:
            P = P.clone() if isinstance(P, RingPreds) else sampler._state(P).clone()
        self.P = sampler._initial_preds(self.X, P)  # (pixels are replaced by ring coefficients where those are carried)

        def warm_up():  # `iterate` without `out` leaves X and P as they are
            x, p = self.X, self.P
            for _ in range(2):
                x, p = sampler.iterate(x, p)

        def record():
            for _ in range(self.iterations):
                sampler.iterate(self.X, self.P, out=(self.X, self.P))

        self.dstep = sampler._dstep = torch.full((1,), sampler._step_counter + 1, dtype=torch.int64,
                                                 device=self.X.device)
        try:
            _warm_up(warm_up)
            self.dstep.fill_(sampler._step_counter + 1)  # the warm-up did not happen as far as the chain is concerned
            self.graph = _record_graph(record)
        finally:
            sampler._dstep = None

    def step(self):
        """advance the chain by `iterations` iterations (asynchronous, like any kernel launch)"""
        self.graph.replay()
        self.sampler._step_counter += self.iterations

    def state(self):
        """(X, predictions) as [nchains, .] tensors (ring-carried predictions are converted to pixels)"""
        return self.X, PxMCMC._pix(self.P)

    def _state_raw(self):
        return self.X, self.P

    def release(self):
        """drop the graph and its step counter; X and P stay valid"""
        self.graph = self.dstep = None


class PxMALA(MYULA):
    """MYULA + Metropolis-Hastings correction, optional step-size tuning
    (pxmcmc/mcmc.py:204-289).  The accept decision uses numpy's global RNG after the
    Gaussian draw, as in the reference."""

    def __init__(self, forward, prox, mcmcparams=PxMCMCParams(), tune_delta=True, **kw):
        super().__init__(forward, prox, mcmcparams, **kw)
        self.tune_delta = tune_delta
        if self.nchains != 1 and not self._device_resident():
            raise NotImplementedError("batched PxMALA chains need the device-resident loop: noise='device', a native "
                                      "operator with a diagonal covariance and an L1 prior")

    def _logtrans_dev(self, X1, X2, proxf, gradg):
        s = complex(D.to_host(self._transition_sums(X1, X2, proxf, gradg))[0])
        return -(1 / 2 * self.delta) * s ** 2

    def calc_logtransition(self, X1, X2, proxf, gradg):
        """log q(X2|X1) exactly as the reference codes it (pxmcmc/mcmc.py:281-289)"""
        val = self._logtrans_dev(self._state(X1), self._state(X2), self._state(proxf), self._state(gradg))
        return val if np.iscomplexobj(X1) or np.iscomplexobj(X2) or np.iscomplexobj(proxf) or np.iscomplexobj(gradg) or D.is_dev(X1) else val.real

    def _device_resident(self):
        """True when an iteration can run without a host round trip: Philox noise, a native operator with a
        diagonal covariance and a native L1 prior, one chain"""
        return (self.noise == "device" and getattr(self.forward, "_pxm_native", False)
                and getattr(self.forward, "_diag", None) is not None and is_library_l1(self.prior)
                and getattr(self.forward, "_pxm_allreduce", None) is None)

    trace_ring = 1 << 16  # slots of the device-side acceptance / step-size trace rings (drained to the host when full)

    def _run_device(self, start_point=None, checkpoint=None, checkpoint_every=0, resume=None):
        """The same loop with the accept test on the device (`pxm_pxmala_accept`): the step size, log pi(Xc) and the
        traces live in device memory, the accepted proposal is copied over the state by a predicated kernel, and the
        host reads the decision only on the thinning grid (where the reference stores accepted samples).  The traces
        are rings of `trace_ring` slots drained to the host every `trace_ring` iterations, so a run may be as long as
        the reference's (nburn = 10^7 in experiments/weaklensing/main.py:110-119)."""
        dv = D.dev()
        nch = self.nchains
        cap = int(self.trace_ring)
        acc_chunks, dl_chunks = [], []  # drained parts of the traces: [nch, cap] each
        i = 0
        js = np.zeros(nch, dtype=np.int64)  # tracked samples per chain (accepted proposals on the thinning grid)
        self._stats_begin()
        if resume is not None:
            ck = self._load_ckpt(resume)
            i, js = int(ck["i"]), ck["js"].astype(np.int64)
            X_curr, curr_preds = self._state(ck["X"]), self._state(ck["P"])
            acc_chunks, dl_chunks = [ck["acc_done"]], [ck["dl_done"]]
            delta0 = float(ck["delta0"])
        else:
            X_curr, curr_preds = self._initial_sample(start_point)
            delta0 = self.delta
        X_curr, curr_preds = X_curr.clone(), curr_preds.clone()
        # gradient, prox and log pi of the current state are functions of (X, preds): recomputed (bit-identical) on resume
        gradg_curr = D.to_dev_c(self._gradg_dev(curr_preds)).clone()
        proxf_curr = D.to_dev_c(self._proxf_dev(X_curr)).clone()
        if resume is not None:
            S = torch.from_numpy(np.ascontiguousarray(ck["S"])).to(dv)
        else:
            lp, l2, pr = self._logpi_dev(X_curr, curr_preds)
            S = np.zeros((nch, 16))
            S[:, 0], S[:, 1], S[:, 2], S[:, 3] = self.delta, 1 - self.delta / self.lmda, self.delta / self.lmda, np.sqrt(2 * self.delta)
            S[:, 4], S[:, 5], S[:, 6], S[:, 7], S[:, 8] = np.real(lp), np.imag(lp), np.real(l2), np.imag(l2), pr
            S = torch.from_numpy(S).to(dv)
        acc = torch.zeros((nch, cap), dtype=torch.int8, device=dv)
        dl = torch.zeros((nch, cap + 1), dtype=D.FDT, device=dv)
        mode = 3 if self.complex else 2
        cur = [X_curr, curr_preds, gradg_curr, proxf_curr]

        def drain(upto):
            """move the first `upto` ring slots (iterations i - upto .. i - 1) to the host lists"""
            if upto:
                acc_chunks.append(acc[:, :upto].cpu().numpy())
                dl_chunks.append(dl[:, 1: upto + 1].cpu().numpy())

        def traces():
            a = np.concatenate(acc_chunks, axis=1) if acc_chunks else np.zeros((nch, 0), dtype=np.int8)
            d = np.concatenate(dl_chunks, axis=1) if dl_chunks else np.zeros((nch, 0))
            return a, d

        def body(i_arg, step_arg):
            """one iteration; (i_arg, step_arg) = (-1, 0): iteration index and Philox step come from S[:, 13], S[:, 14]"""
            X_prop = D.myula_update_dpar_dev(cur[0], cur[3], cur[2], None, 0.0, S, mode, self.seed, step_arg, self.stream0)
            prop_preds = D.to_dev_c(self._forward_dev(X_prop))
            gradg_prop = D.to_dev_c(self._gradg_dev(prop_preds))
            proxf_prop = D.to_dev_c(self._proxf_dev(X_prop))
            L2p, priorp = self._logpi_terms_dev(X_prop, prop_preds)
            s1 = D.reduce_dpar_dev(cur[0], X_prop, cur[3], cur[2], S, self.lmda)
            s2 = D.reduce_dpar_dev(X_prop, cur[0], proxf_prop, gradg_prop, S, self.lmda)
            # priorp is the real view of a complex reduction result: same address, the kernel reads its real part
            D.pxmala_accept_dev(S, s1, s2, L2p, priorp, self.mu, self.lmda, self.tune_delta, i_arg, self.seed, step_arg,
                                self.stream0, acc, dl)
            D.select_if_dev(S, cur, [X_prop, prop_preds, gradg_prop, proxf_prop])

        # One CUDA graph per iteration (~30 launches otherwise issued one by one from Python): the first iterations
        # run eagerly (they warm up tables, lazy uploads and allocator pools, and ARE iterations of the chain), then the
        # iteration is captured with its counters in the state blocks
        graph = None
        i_graph = i + 2 if self._graphed() else None

        def after(i):
            on_grid = self._on_grid(i)
            verbose = self.verbosity > 0 and (i + 1) % self.verbosity == 0
            if on_grid or verbose:
                st = S.cpu().numpy()  # the only host synchronisation
                take = [c for c in range(nch) if on_grid and st[c, 9] != 0.0 and js[c] < self.nsamples]
                if take and (self._stats is not None or self._cred is not None):  # own sample index, -1: none now
                    jd = np.full(nch, -1, dtype=np.int64)
                    jd[take] = js[take]
                    self._stats_push(cur[0], cur[1], d_j=torch.from_numpy(jd).to(dv), nactive=len(take))
                if take:
                    Xh = D.to_host(cur[0]) if hasattr(self, "chain") else None
                    Ph = D.to_host(cur[1]) if hasattr(self, "preds") else None
                    for c in take:
                        j = int(js[c])
                        if hasattr(self, "logPi"):
                            self._put(self.logPi, j, complex(st[c, 4], st[c, 5]), c)
                        if hasattr(self, "L2s"):
                            self._put(self.L2s, j, complex(st[c, 6], st[c, 7]), c)
                        if hasattr(self, "priors"):
                            self._put(self.priors, j, st[c, 8], c)
                        if Ph is not None:
                            self._put(self.preds, j, Ph[c], c)
                        if Xh is not None:
                            self._put(self.chain, j, Xh[c], c)
                        js[c] += 1
                if verbose:
                    done = sum(int(a.sum()) for a in acc_chunks) + int(acc[:, : (i % cap) + 1].sum().item())
                    self._print_progress(int(js[0]) - 1, st[0, 4], L2=st[0, 6], prior=st[0, 8],
                                         acceptanceRate=done / float(nch * (i + 1)))

        def save(i_next):
            a, d = traces()
            part = i_next % cap
            if part:
                a = np.concatenate([a, acc[:, :part].cpu().numpy()], axis=1)
                d = np.concatenate([d, dl[:, 1: part + 1].cpu().numpy()], axis=1)
            self._save_ckpt(checkpoint, i=i_next, js=js, X=D.to_host(cur[0]), P=D.to_host(cur[1]), S=S.cpu().numpy(),
                            acc_done=a, dl_done=d, delta0=delta0)

        if resume is not None and i % cap:
            # the ring is addressed by i mod cap: put the undrained tail of the restored traces back in its slots
            part = i % cap
            a, d = acc_chunks.pop(), dl_chunks.pop()
            acc[:, :part] = torch.from_numpy(np.ascontiguousarray(a[:, a.shape[1] - part:])).to(dv)
            dl[:, 1: part + 1] = torch.from_numpy(np.ascontiguousarray(d[:, d.shape[1] - part:])).to(dv)
            if a.shape[1] > part:
                acc_chunks.append(a[:, : a.shape[1] - part])
                dl_chunks.append(d[:, : d.shape[1] - part])

        while js.min() < self.nsamples:
            self._step_counter += 1
            if i == i_graph:
                S[:, 13], S[:, 14] = float(i), float(self._step_counter)
                graph = _record_graph(lambda: body(-1, 0))
            if graph is not None:
                graph.replay()
            else:
                body(i, self._step_counter)
            after(i)
            i += 1
            if i % cap == 0:
                drain(cap)
            if checkpoint is not None and checkpoint_every and i % checkpoint_every == 0:
                save(i)
        if checkpoint is not None:
            save(i)
        drain(i % cap)
        X_curr, curr_preds = cur[0], cur[1]
        at, dt = traces()
        at = at.astype(int)
        first = np.full((nch, 1), delta0)
        dt = np.concatenate([first, dt], axis=1) if self.tune_delta else first
        # one chain: the reference's flat lists; several chains: arrays with a leading chain axis
        self.acceptance_trace = [int(v) for v in at[0]] if nch == 1 else at
        self.deltas_trace = [float(v) for v in dt[0]] if nch == 1 else dt
        self.delta = float(S[0, 0].item())
        self.deltas = S[:, 0].cpu().numpy()
        self._stats_end()
        self._final_state = (X_curr.clone(), curr_preds.clone())
        print("\nDONE")

    def _shared_uniform(self):
        """the uniform of the accept test; the ranks of an m-sharded chain must all use rank 0's draw"""
        u = np.random.rand()
        red = getattr(self.forward, "_pxm_allreduce", None)
        if red is not None:
            import torch.distributed as dist

            mine = u if (not dist.is_initialized() or dist.get_rank() == 0) else 0.0
            u = float(red(torch.tensor([mine], dtype=D.FDT, device=D.dev())).item())
        return u

    def _transition_sums(self, X1, X2, proxf, gradg):
        """sum (X2 - X1 - (delta/2) grad log pi(X1))^2 per chain as a device tensor, summed over the ranks of an m-sharded
        operator BEFORE it is squared again (pxmcmc/mcmc.py:286-289)"""
        s = D.reduce_dev(2, X1, b=X2, c=proxf, d=gradg, delta=self.delta, lmda=self.lmda)
        red = getattr(self.forward, "_pxm_allreduce", None)
        return red(s) if red else s

    def run(self, start_point=None, *, checkpoint=None, checkpoint_every=0, resume=None):
        """the loop of pxmcmc/mcmc.py:218-275.  `checkpoint` / `checkpoint_every` / `resume` as in `MYULA.run`."""
        if self._device_resident():
            return self._run_device(start_point, checkpoint, checkpoint_every, resume)
        self.acceptance_trace = []
        self.deltas_trace = [self.delta]
        i = 0
        j = 0
        self._stats_begin()
        if resume is not None:
            ck = self._load_ckpt(resume)
            i, j = int(ck["i"]), int(ck["j"])
            X_curr, curr_preds = self._state(ck["X"]), self._state(ck["P"])
            self.acceptance_trace = [int(v) for v in ck["acc_done"]]
            self.deltas_trace = [float(v) for v in ck["dl_done"]]
        else:
            X_curr, curr_preds = self._initial_sample(start_point)
        # functions of (X, preds): recomputed (bit-identical) on resume
        gradg_curr = D.to_dev_c(self._gradg_dev(curr_preds))
        proxf_curr = self._proxf_dev(X_curr)
        lp, l2, pr = self._logpi_dev(X_curr, curr_preds)
        logpiXc, L2Xc, priorXc = lp[0], l2[0], pr[0]

        def save(i_next):
            self._save_ckpt(checkpoint, i=i_next, j=j, X=D.to_host(X_curr), P=D.to_host(curr_preds),
                            acc_done=np.asarray(self.acceptance_trace, dtype=np.int8), dl_done=np.asarray(self.deltas_trace))

        while j < self.nsamples:
            X_prop = self._propose_dev(X_curr, proxf_curr, gradg_curr)
            prop_preds = D.to_dev_c(self._forward_dev(X_prop))
            gradg_prop = D.to_dev_c(self._gradg_dev(prop_preds))
            proxf_prop = self._proxf_dev(X_prop)
            terms = self._logpi_terms_dev(X_prop, prop_preds)
            if terms is not None:
                # the four reductions of the accept test leave the device in ONE copy (one host sync per iteration)
                s1 = self._transition_sums(X_curr, X_prop, proxf_curr, gradg_curr)
                s2 = self._transition_sums(X_prop, X_curr, proxf_prop, gradg_prop)
                v = torch.cat([s1, s2, terms[0], terms[1].to(D.CDT)]).cpu().numpy()
                logtransXcXp = -(1 / 2 * self.delta) * complex(v[0]) ** 2
                logtransXpXc = -(1 / 2 * self.delta) * complex(v[1]) ** 2
                L2Xp, priorXp = v[2], v[3].real
                logpiXp = -self.mu * priorXp - L2Xp
            else:
                logtransXcXp = self._logtrans_dev(X_curr, X_prop, proxf_curr, gradg_curr)
                logtransXpXc = self._logtrans_dev(X_prop, X_curr, proxf_prop, gradg_prop)
                lp, l2, pr = self._logpi_dev(X_prop, prop_preds)
                logpiXp, L2Xp, priorXp = lp[0], l2[0], pr[0]
            logalpha = logtransXpXc + logpiXp - logtransXcXp - logpiXc
            accept = _cplx_lt(np.log(self._shared_uniform()), logalpha)
            if accept:
                X_curr, curr_preds, gradg_curr, proxf_curr = X_prop, prop_preds, gradg_prop, proxf_prop
                logpiXc, L2Xc, priorXc = logpiXp, L2Xp, priorXp
                self.acceptance_trace.append(1)
            else:
                self.acceptance_trace.append(0)
            if self.tune_delta:
                self._tune_delta(i)
                self.deltas_trace.append(self.delta)
            if self._on_grid(i) and accept:
                self._tracking(j, X_curr, curr_preds, [logpiXc], [L2Xc], [priorXc])
                self._stats_push(X_curr, curr_preds, j)
                j += 1
            if self.verbosity > 0 and (i + 1) % self.verbosity == 0:
                self._print_progress(j - 1, np.real(logpiXc), L2=np.real(L2Xc), prior=priorXc,
                                     acceptanceRate=np.mean(self.acceptance_trace))
            i += 1
            if checkpoint is not None and checkpoint_every and i % checkpoint_every == 0:
                save(i)
        if checkpoint is not None:
            save(i)
        self._stats_end()
        self._final_state = (X_curr, curr_preds)
        print("\nDONE")

    def _tune_delta(self, i):
        """pxmcmc/mcmc.py:277-279"""
        delta = self.delta * (1 + (self.acceptance_trace[i] - 0.5) / ((i + 1) ** 0.75))
        self.delta = min(max(delta, self.lmda * 1e-8), self.lmda / 2)


class SKROCK(PxMCMC):
    """Stochastic orthogonal Runge-Kutta-Chebyshev sampler (pxmcmc/mcmc.py:292-383).
    The reference evaluates K_s by naive recursion (4 059 gradient evaluations at
    s=10); K_0..K_s are evaluated bottom-up here (s evaluations, identical values).

    `scheme` (keyword-only):
    * "reference" (default): the recursion exactly as the reference codes it (ratio T_{j-1}(omega_0) / T_j(omega_1), a
      scalar k_j = 1 added and K_{j-2} subtracted).  It reproduces the reference's chains, but its step multiplies the
      state by about 1e8 at s = 10 whatever the step size: it does not sample.
    * "published": SK-ROCK of Abdulle, Almuslimani & Vilmart (2018), as used by Pereyra, Vargas-Mieles & Zygalakis
      (2020): K_j = mu_j delta grad log pi(K_{j-1}) + nu_j K_{j-1} + kappa_j K_{j-2} with the ratio
      T_{j-1}(omega_0) / T_j(omega_0) and kappa_j = 1 - nu_j.  Stable for step sizes up to `stability_limit` / Lip,
      about s^2 times MYULA's."""

    def __init__(self, forward, prox, mcmcparams=PxMCMCParams(), *, scheme="reference", **kw):
        if scheme not in ("reference", "published"):
            raise ValueError(f"scheme must be 'reference' or 'published', got {scheme!r}")
        self._scheme = scheme
        super().__init__(forward, prox, mcmcparams=mcmcparams, **kw)
        self.eta = 0.05
        self.omega_0 = 1 + self.eta / (self.s * self.s)
        self.omega_1 = chebyshev1(self.omega_0, self.s) / cheb1der(self.omega_0, self.s)
        self._recursion_coefs()

    @property
    def scheme(self):
        """"reference" or "published" (read-only: the coefficients are fixed at construction)"""
        return self._scheme

    @property
    def stability_limit(self):
        """(omega_0 + 1) / omega_1: the published scheme is stable (|R(p)| <= 1, R(p) = T_s(omega_0 - omega_1 p) /
        T_s(omega_0) the step's deterministic factor) for p = delta * Lip(grad log pi_lambda) <= stability_limit, where
        Lip >= 1 / lmda from the Moreau-Yosida term.  17.4 at s = 3, 48.4 at s = 5, 193.6 at s = 10 (the bound usually
        quoted, (s - 1/2)^2 (2 - 4 eta / 3) - 3/2, is a conservative version of it).  At it |R| = 1 / T_s(omega_0); |R|
        passes 1 at 2 omega_0 / omega_1, (omega_0 - 1) / omega_1 further.  NaN for the
        reference scheme, which is stable for no step size."""
        return (self.omega_0 + 1) / self.omega_1 if self._scheme == "published" else float("nan")

    def _save_ckpt(self, path, **fields):
        super()._save_ckpt(path, scheme=self._scheme, **fields)

    def _load_ckpt(self, path):
        with np.load(path if path.endswith(".npz") else path + ".npz", allow_pickle=False) as f:
            scheme = str(f["scheme"]) if "scheme" in f.files else "reference"  # files written before the option
        if scheme != self._scheme:
            raise ValueError(f"checkpoint was written by a SKROCK sampler with scheme={scheme!r}, not {self._scheme!r}")
        return super()._load_ckpt(path)

    def _initial_preds(self, Xd, P=None):
        """pixels whatever the operator: the stage gradients are taken at other points than the state (`_gradg_at`),
        so nothing consumes ring coefficients of the state"""
        return D.to_dev_c(self._forward_dev(Xd)) if P is None else P

    def iterate(self, X_curr, curr_preds, out=None):
        """one step and the predictions of the new state on device tensors [nchains, .] (the step itself does not read
        `curr_preds`).  `out = (X_buf, P_buf)` as in `MYULA.iterate`: the input buffers themselves are allowed, which
        is how captured graphs advance in place."""
        if out is None:
            X_new = self._chain_step_dev(X_curr)
            return X_new, D.to_dev_c(self._forward_dev(X_new))
        X_new = self._chain_step_dev(X_curr, out=out[0])
        return X_new, self._forward_dev(X_new, out=out[1])

    def _chain_step_dev(self, Xd, Z=None, out=None):
        """Z: real [nchains, n] normals, a (real, imaginary) pair when `complex` (pxmcmc/mcmc.py:344-347), or a
        `device.SkrockNoise`; None draws it (host RNG, or Philox normals regenerated inside the stage kernels)"""
        n = Xd.shape[-1]
        nch = Xd.shape[0]
        dstep = None
        if Z is None:
            if self.noise == "device":  # Philox normals, step counter on the host or (graph replays) on the device
                dstep = getattr(self, "_dstep", None)
                if dstep is None:
                    self._step_counter += 1
                # complex: one draw of 2n normals per chain, the first n the real, the last n the imaginary parts
                Z = D.SkrockNoise(complex=self.complex, seed=self.seed, step=self._step_counter, stream0=self.stream0,
                                  dstep=dstep)
            else:
                Z = D.to_dev_f(np.random.randn(n * nch)).reshape(Xd.shape)
                if self.complex:  # the reference's order: real part, then imaginary part
                    Z = (Z, D.to_dev_f(np.random.randn(n * nch)).reshape(Xd.shape))
        if not isinstance(Z, D.SkrockNoise):
            Z = D.SkrockNoise(*Z) if isinstance(Z, tuple) else D.SkrockNoise(Z)
        out = self._K_recursion(Xd, self.s, Z, out=out)
        if dstep is not None:
            D.check(D.lib.pxm_counter_add(D.ptr(dstep), 1, D.stream_ptr()))
        return out

    def chain_step(self, X):
        """one SKROCK step (pxmcmc/mcmc.py:338-347)"""
        out = self._chain_step_dev(self._state(X))
        return out if D.is_dev(X) else D.to_host(out[0])

    def _K_recursion(self, Xd, s, Z, out=None):
        """K_s of pxmcmc/mcmc.py:349-368, memoised, one fused kernel per stage (and the shift Y = X + nu_1 sqrt(2 delta) Z
        the first gradient is evaluated at).  Z: a `device.SkrockNoise`.  `out` (may be Xd) receives K_s."""
        if s == 0:
            return Xd if out is None else D.copy_into(out, Xd)
        sq = np.sqrt(2 * self.delta)
        Y = D.skrock_shift_dev(Xd, self.nus[1] * sq, Z)
        K_prev = D.skrock_stage_dev(Xd, None, *self._stage_inputs(Y), self.lmda, self.mus[1] * self.delta, 1.0, 0.0, 0.0,
                                    Z=Z, c_shift=self.nus[1] * sq, e=self.ks[1] * sq, out=out if s == 1 else None)
        K_prev2 = Xd
        for j in range(2, s + 1):
            # reference: ... + nu_j K_{j-1} + k_j - K_{j-2};  published: ... + nu_j K_{j-1} + kappa_j K_{j-2}
            c, c0 = (-1.0, self.ks[j]) if self._scheme == "reference" else (self.ks[j], 0.0)
            K = D.skrock_stage_dev(K_prev, K_prev2, *self._stage_inputs(K_prev), self.lmda, self.mus[j] * self.delta,
                                   self.nus[j], c, c0, out=out if j == s else None)
            K_prev2, K_prev = K_prev, K
        return K_prev

    def _stage_inputs(self, P):
        """(gradg, prox, Tvec, Tscalar) of grad log pi at P for the stage kernel: the soft threshold is applied inside
        it when the prior allows, else prox(P) is given"""
        gradg = self._gradg_at(P)
        fused = self._fused_prox()
        if fused is not None:
            return gradg, None, fused[0], fused[1]
        return gradg, self._proxf_dev(P), None, 0.0

    def _recursion_coefs(self):
        """mu_j, nu_j and k_j (reference, exactly as pxmcmc/mcmc.py:370-383 computes them) or kappa_j (published);
        stage 1 is the same in both schemes"""
        self.mus = np.zeros(self.s + 1)
        self.nus = np.zeros(self.s + 1)
        self.ks = np.zeros(self.s + 1)
        self.mus[1] = self.omega_1 / self.omega_0
        self.nus[1] = self.s * self.omega_1 / 2
        self.ks[1] = self.s * self.omega_1 / self.omega_0
        for j in range(2, self.s + 1):
            if self._scheme == "reference":
                cheb_ratio = chebyshev1(self.omega_0, j - 1) / chebyshev1(self.omega_1, j)
            else:
                cheb_ratio = chebyshev1(self.omega_0, j - 1) / chebyshev1(self.omega_0, j)
            self.mus[j] = 2 * self.omega_1 * cheb_ratio
            self.nus[j] = 2 * self.omega_0 * cheb_ratio
            self.ks[j] = 1 - self.nus[0] if self._scheme == "reference" else 1 - self.nus[j]
