"""Forward operators mirroring ``pxmcmc/forward.py`` of the reference."""
import numpy as np
from scipy import sparse

from . import device as D
from .measurements import Identity, PathIntegral
from .transforms import SphericalWaveletTransform
from .utils import mw_size


class RingPreds:
    """Predictions of an Identity-measurement synthesis operator kept in the transform's own intermediate space instead
    of pixels: `kind == "ring"`: ring-Fourier coefficients F_m(theta_t) of the image (the plan's ring array);
    `kind == "harm"`: its harmonic coefficients f_lm (the plan's harmonic array).  What `ForwardOperator.forward_ring`
    returns and `gradg_from_ring` consumes.  `.pixels()` gives the ordinary [nchains, npix] predictions."""

    __slots__ = ("t", "op", "nb", "kind")

    def __init__(self, t, op, nb, kind="ring"):
        self.t, self.op, self.nb, self.kind = t, op, int(nb), kind

    def pixels(self):
        return self.op.ring_to_pixels(self)

    def clone(self):
        return RingPreds(self.t.clone(), self.op, self.nb, self.kind)

    def scaled_(self, c):
        self.t.mul_(c)
        return self


class ForwardOperator:
    """Transform + measurement + Gaussian data fidelity (pxmcmc/forward.py:9-88).

    ``forward`` / ``calc_gradg`` take a numpy vector (numpy out) or a CUDA tensor
    [n] / [nchains, n] (tensor out).  ``invcov`` is kept as the scipy sparse matrix
    the reference builds; the device path uses its diagonal.
    """

    def __init__(self, data, sig_d, setting, transform=None, measurement=None, nparams=None):
        self.data = data
        self.invcov = self._build_inverse_covariance_matrix(sig_d)
        if setting not in ["analysis", "synthesis"]:
            raise ValueError
        self.setting = setting
        if transform is not None:
            self.transform = transform
        if measurement is not None:
            self.measurement = measurement
        if nparams is not None:
            self.nparams = nparams
        self._dev = None

    # ------------------------------------------------------------------ device state
    @property
    def _pxm_native(self):
        return getattr(getattr(self, "transform", None), "_pxm_native", False) and getattr(
            getattr(self, "measurement", None), "_pxm_native", False
        ) and self._diag is not None

    def _upload(self):
        if self._dev is None:
            if self._diag is None:
                raise NotImplementedError("a full covariance matrix is not supported on the device path")
            self._dev = (D.to_dev_c(np.asarray(self.data).ravel()), D.to_dev_c(self._diag))
        return self._dev

    # ------------------------------------------------------------------ public API
    def forward(self, X):
        """data predictions of sample X (pxmcmc/forward.py:36-46)"""
        if self.setting == "analysis":
            return self._forward_analysis(X)
        return self._forward_synthesis(X)

    def calc_gradg(self, preds):
        """gradient of the Gaussian data fidelity (pxmcmc/forward.py:48-58)"""
        if self.setting == "analysis":
            return self._gradg_analysis(preds)
        return self._gradg_synthesis(preds)

    def _forward_analysis(self, X):
        return self.measurement.forward(X)

    # Weak lensing behind a wavelet synthesis: Psi ends with A_inv(L,0) and the measurement starts with A_fwd(L,0);
    # A_fwd o A_inv = I on f_lm (MW sampling is exact), so the two full-L transforms of each direction are skipped
    # (SURVEY.md 3.5; same result to round-off, a third of the Legendre tables never streamed).  Set
    # `fuse_harmonic = False` for the reference's literal composition.
    fuse_harmonic = True

    def _fused(self):
        t, m = getattr(self, "transform", None), getattr(self, "measurement", None)
        return (self.fuse_harmonic and self.setting == "synthesis" and getattr(m, "_pxm_harmonic_input", False)
                and (type(m).forward, type(m).adjoint) == getattr(type(m), "_pxm_fused_methods", None)  # not overridden
                and hasattr(t, "_inverse_harmonic") and getattr(t, "spin", 0) == 0 and getattr(t, "L", None) == getattr(m, "L", -1))

    # Identity measurement behind a wavelet synthesis: Psi ends with the ring FFT F -> pixels and the gradient of the next
    # iteration starts with the ring FFT pixels -> F.  The DFT of length 2L-1 is invertible, so when the inverse
    # covariance is constant along every ring (a scalar sigma, or the reference's per-ring noise sqrt(sigma^2 / area),
    # experiments/earthtopography/main.py:92-94) the pair cancels: FFT_in(ic (FFT_out(F) - d)) = ic_t ((2L-1) F - FFT_in(d)).
    # The samplers then carry the predictions as ring coefficients (`RingPreds`) and convert them to pixels only where
    # pixels are needed (tracked samples, checkpoints, the host-buffer path).  Same results to round-off;
    # `fuse_ring = False` restores the literal composition.
    # When the inverse covariance is ONE constant over the whole sphere (a scalar sigma) the same composition collapses
    # further, per order m, to g = ic (G f - b) with the Gram matrix G^m = (2L-1) Lambda^T Lambda and b = A_inv^dagger(data)
    # (pxm_wav_gram_gradient): one contraction instead of the two full-L ones; the predictions are then carried as f_lm.
    fuse_ring = True
    fuse_gram = True

    def _ring_kind(self):
        """'harm' (Gram form), 'ring', or None"""
        if not self._ring_fusable():
            return None
        if self.fuse_gram and self._gram_weights() is not False:
            return "harm"
        return "ring"

    def _gram_weights(self):
        """How the Gram form applies: None -- the inverse covariance is ONE constant c (G = n Lambda^T Lambda, g = c (G f - b));
        (phase, w) -- it is constant along every ring with a common complex phase, ic_t = phase * w_t with w_t real
        (the reference's per-ring noise levels, experiments/earthtopography/main.py:92-94; a complex data vector turns
        the real variances into var (1 + i) / sqrt 2, pxmcmc/forward.py:80-82: a common phase): G = n Lambda^T diag(w) Lambda,
        g = phase (G f - A_inv^dagger(w d)); False -- it does not (the phases differ)"""
        c = getattr(self, "_gram_w_cache", None)
        if c is None or c[0] is not self._diag:
            d = np.asarray(self._diag)
            if bool(np.all(d == d[0])):
                r = None
            else:
                L = self.transform.L
                ring = d.reshape(L, 2 * L - 1)[:, 0]
                phase = ring[0] / abs(ring[0])
                w = ring / phase
                r = (complex(phase), np.ascontiguousarray(w.real)) if bool(np.all(np.abs(w.imag) <= 1e-13 * np.abs(w.real))) else False
            self._gram_w_cache = c = (self._diag, r)
        return c[1]

    def _own_methods(self):
        """True unless a user subclass overrides the methods the carried forms stand in for (it is then not bypassed)"""
        return all(getattr(type(self), n) is getattr(ForwardOperator, n)
                   for n in ("forward", "calc_gradg", "_forward_synthesis", "_gradg_synthesis", "_residual"))

    def _ring_fusable(self):
        t, m = getattr(self, "transform", None), getattr(self, "measurement", None)
        if not (self.fuse_ring and self.setting == "synthesis" and self._diag is not None and self._own_methods()):
            return False
        if type(m) is not Identity or m.ndata != m.npix:
            return False
        if (type(t).inverse is not SphericalWaveletTransform.inverse
                or type(t).inverse_adjoint is not SphericalWaveletTransform.inverse_adjoint or not hasattr(t, "_plan")):
            return False
        if len(self._diag) != t.L * (2 * t.L - 1):
            return False
        return self._ic_rings() is not None

    def _ic_rings(self):
        """inverse covariance of every ring as a complex device vector [L], or None when it varies along a ring"""
        c = getattr(self, "_ic_rings_cache", None)
        if c is None or c[0] is not self._diag:
            L = self.transform.L
            d = np.asarray(self._diag).reshape(L, 2 * L - 1)
            # constant along every ring up to rounding: the reference's own per-ring noise levels come out of
            # calc_pixel_areas with last-bit differences along phi (pxmcmc/utils.py:227-246)
            ok = bool(np.all(np.abs(d - d[:, :1]) <= 1e-13 * np.abs(d[:, :1])))
            self._ic_rings_cache = c = (self._diag, D.to_dev_c(np.ascontiguousarray(d[:, 0])) if ok else None)
        return c[1]

    def _ring_data(self, nb):
        c = getattr(self, "_ring_data_cache", None)
        if c is None:
            c = self._ring_data_cache = {}
        if nb not in c:
            data_d, _ = self._upload()
            c[nb] = self.transform._plan(nb).pix_to_ring(data_d.reshape(1, -1))
        return c[nb]

    def forward_ring(self, X, out=None):
        """predictions of the state(s) as ring coefficients (synthesis without its last ring FFT)"""
        x = D.to_dev_c(X)
        x = x.unsqueeze(0) if x.dim() == 1 else x
        nb = x.shape[0]
        kind = out.kind if out is not None else self._ring_kind()
        plan = self.transform._plan(nb)
        if kind == "harm":
            t = plan.synthesis_to_harm(x, out=None if out is None else out.t)
        else:
            t = plan.synthesis_to_ring(x, out=None if out is None else out.t)
        return out if out is not None else RingPreds(t, self, nb, kind)

    def _harm_b(self, nb):
        c = getattr(self, "_harm_b_cache", None)
        if c is None:
            c = self._harm_b_cache = {}
        if nb not in c:
            data_d, _ = self._upload()
            gw = self._gram_weights()
            if gw:  # per-ring weights: b = A_inv^dagger(w d)
                L = self.transform.L
                wpix = D.to_dev_c(np.repeat(gw[1], 2 * L - 1).astype(complex))
                data_d = data_d * wpix
            c[nb] = self.transform._plan(nb).pix_to_harm_adjoint(data_d.reshape(1, -1))
        return c[nb]

    def gradg_from_ring(self, R):
        """gradient of the data fidelity from ring- / harmonic-space predictions"""
        plan = self.transform._plan(R.nb)
        if R.kind == "harm":
            gw = self._gram_weights()
            # the plan's Gram table carries this operator's ring weights (regenerated, ~1 ms, when another operator
            # sharing the transform object has put its own there since)
            key = None if not gw else (id(self._diag), len(gw[1]))
            if plan.gram_key != key:
                plan.set_gram_weights(None if not gw else gw[1], key)
            ic = complex(np.asarray(self._diag)[0]) if not gw else gw[0]
            return plan.gram_gradient(R.t, self._harm_b(R.nb), ic, R.nb)
        resid = plan.ring_resid(R.t, self._ring_data(R.nb), self._ic_rings(), R.nb)
        return plan.synthesis_adjoint_from_ring(resid, R.nb)

    def ring_to_pixels(self, R):
        plan = self.transform._plan(R.nb)
        return plan.harm_to_pix(R.t, R.nb) if R.kind == "harm" else plan.ring_to_pix(R.t, R.nb)

    def pixels_to_ring(self, P):
        """ring form of pixel predictions (the harmonic form cannot be recovered from pixels without the analysis
        tables: callers recompute it from the state with `forward_ring`)"""
        p = D.to_dev_c(P)
        p = p.unsqueeze(0) if p.dim() == 1 else p
        plan = self.transform._plan(p.shape[0])
        return RingPreds(plan.pix_to_ring(p), self, p.shape[0], "ring").scaled_(1.0 / (2 * self.transform.L - 1))

    # Two REAL-valued chains as one complex chain (MYULA(real_pairs=True)).  With real data and a real inverse
    # covariance every linear map of the synthesis path (ring FFTs, Legendre contractions, the data-fidelity residual) is
    # complex-linear AND maps real fields to real fields, so z = x_a + i x_b travels through it as (result_a) + i (result_b):
    # the transforms of two chains for the price of one.  The reference computes the same real chain in complex
    # arithmetic with a zero imaginary part (pys2let returns complex arrays, experiments/earthtopography/main.py:80-123).
    # Both chains see the same data d, i.e. the packed problem has the data (1 + i) d.
    def _pairable(self):
        """None when two real chains may be packed into one complex chain, else the reason why not"""
        t, m = getattr(self, "transform", None), getattr(self, "measurement", None)
        if self.setting != "synthesis" or self._diag is None:
            return "real chain pairs need the synthesis setting and a diagonal covariance"
        if not self._own_methods():
            return "real chain pairs need the library's forward / calc_gradg (a subclass overrides them)"
        if type(m) is not Identity:
            return "real chain pairs need the Identity measurement"
        if (type(t).inverse is not SphericalWaveletTransform.inverse
                or type(t).inverse_adjoint is not SphericalWaveletTransform.inverse_adjoint or not hasattr(t, "_plan")):
            return "real chain pairs need the library's axisymmetric wavelet synthesis (a real operator)"
        if np.iscomplexobj(self.data) or np.any(np.asarray(self._diag).imag != 0):
            return "real chain pairs need real data and a real noise level"
        return None

    def paired(self):
        """the operator of the packed problem: same transform and measurement objects, data (1 + i) d"""
        why = self._pairable()
        if why is not None:
            raise ValueError(why)
        import copy

        op = copy.copy(self)
        op.data = np.asarray(self.data, dtype=float) * (1.0 + 1.0j)
        op._dev = None
        for c in ("_ring_data_cache", "_harm_b_cache", "_ic_rings_cache"):
            if hasattr(op, c):
                delattr(op, c)
        op._is_paired = True
        return op

    # ------------------------------------------------------------------ Lipschitz constant of the data-fidelity gradient
    def _real_positive_ic(self):
        """None when the inverse covariance is diagonal, real and positive (the data fidelity is then the real
        quadratic 1/2 (Phi Psi x - d)^dagger IC (Phi Psi x - d) and gradg its gradient), else the reason why not"""
        if self._diag is None:
            return None
        d = np.asarray(self._diag)
        if np.any(d.imag != 0) or np.any(d.real <= 0):
            return ("the inverse covariance is not real and positive, so gradg is not the gradient of a real data "
                    "fidelity (a real sigma with complex data is turned into the variance var (1 + i) / sqrt 2, "
                    "pxmcmc/forward.py:80-82); pass sigma as a complex array (np.asarray(sigma, dtype=complex)) to skip "
                    "that rule")
        return None

    def _zero_data(self):
        """shadow copy with zero data (same transform, measurement and covariance; data-dependent caches dropped, as in
        `paired`): its gradg is the linear part Psi^dagger Phi^dagger IC Phi Psi of this operator's"""
        import copy

        op = copy.copy(self)
        op.data = np.zeros_like(np.asarray(self.data))
        op._dev = None
        for c in ("_ring_data_cache", "_harm_b_cache", "_ic_rings_cache"):
            if hasattr(op, c):
                delattr(op, c)
        return op

    def _normal_apply(self, X):
        """gradg(forward(X)) through the library's device path: the carried ring / Gram form when it applies, else
        forward + calc_gradg (X: [nchains, n] complex device tensor)"""
        if self._pxm_native and self._ring_fusable():
            return self.gradg_from_ring(self.forward_ring(X))
        if self._pxm_native:
            return D.to_dev_c(self.calc_gradg(self.forward(X)))
        x = D.to_host(X)
        return D.to_dev_c(np.stack([np.asarray(self.calc_gradg(self.forward(v))) for v in x]))

    def lipschitz(self, tol=1e-10):
        """L_f = lambda_max(Psi^dagger Phi^dagger IC Phi Psi): the Lipschitz constant of gradg, the largest eigenvalue of
        its linear part, by ARPACK (scipy.sparse.linalg.eigsh, which="LA", relative accuracy `tol`) with the library's
        own device path as the matrix-vector product (on a zero-data copy of this operator).  Cached per inverse
        covariance.  Synthesis setting with a real, positive, diagonal inverse covariance only (ValueError /
        NotImplementedError with the reason otherwise)."""
        if self.setting != "synthesis":
            raise NotImplementedError("lipschitz: the synthesis setting only")
        if self._diag is None:
            raise NotImplementedError("lipschitz: a full covariance matrix is not supported (diagonal covariances only)")
        if getattr(self, "_pxm_allreduce", None) is not None:
            raise NotImplementedError("lipschitz: m-sharded operators are not supported")
        why = self._real_positive_ic()
        if why is not None:
            raise ValueError("lipschitz: " + why)
        c = getattr(self, "_lipschitz_cache", None)
        if c is not None and c[0] is self._diag and c[1] <= tol:
            return c[2]
        from scipy.sparse.linalg import LinearOperator, eigsh

        op = self._zero_data()
        n = int(self.nparams)
        counter = [0]

        def matvec(v):
            counter[0] += 1
            return D.to_host(op._normal_apply(D.to_dev_c(np.ravel(v)).reshape(1, n))[0])

        A = LinearOperator((n, n), matvec=matvec, dtype=np.complex128)
        v0 = np.random.default_rng(0).standard_normal(n).astype(np.complex128)
        lam = float(eigsh(A, k=1, which="LA", tol=tol, v0=v0, return_eigenvectors=False)[0])
        self._lipschitz_cache = (self._diag, float(tol), lam, counter[0])
        return lam

    def _forward_synthesis(self, X):
        if self._fused():
            return self.measurement._forward_from_harmonic(self.transform._inverse_harmonic(X))
        return self.measurement.forward(self.transform.inverse(X))

    def _residual(self, preds):
        """invcov @ (preds - data) as a dense vector (pxmcmc/forward.py:67-69)"""
        if self._diag is None:  # general covariance: host, as the reference does it
            p = D.to_host(preds) if D.is_dev(preds) else np.asarray(preds)
            r = np.asarray(self.invcov @ (p - np.asarray(self.data))).ravel()
            return D.to_dev_c(r) if D.is_dev(preds) else r
        data_d, ic_d = self._upload()
        return D.like_input(D.resid_dev(D.to_dev_c(preds), data_d, ic_d), preds)

    def _gradg_analysis(self, preds):
        return self.measurement.adjoint(self._residual(preds))

    def _gradg_synthesis(self, preds):
        if self._fused():
            return self.transform._inverse_adjoint_harmonic(self.measurement._adjoint_to_harmonic(self._residual(preds)))
        return self.transform.inverse_adjoint(self._gradg_analysis(preds))

    def _build_inverse_covariance_matrix(self, sig_d):
        """scalar / vector / matrix sigma -> sparse inverse covariance
        (pxmcmc/forward.py:74-88), including the reference's rule that a real
        variance paired with complex data becomes var*(1+i)/sqrt(2)."""
        self._diag = None
        if isinstance(sig_d, np.ndarray) and len(sig_d.shape) == 2:
            if sig_d.shape[0] != sig_d.shape[1]:
                raise ValueError("Covariance matrix should be square")
            from scipy.sparse import linalg as sla

            return sla.inv(sig_d)
        var = sig_d ** 2
        if np.iscomplexobj(self.data) and not np.iscomplexobj(var):
            var = var / np.sqrt(2) * (1 + 1j)
        ndata = len(self.data)
        if isinstance(var, (float, int, complex)):
            self._diag = np.full(ndata, 1 / var, dtype=complex)
            return sparse.identity(ndata).dot(1 / var)
        if var.size == ndata and len(var.shape) == 1:
            self._diag = (1 / var).astype(complex)
            return sparse.diags(1 / var)
        raise TypeError("sig_d must be a float scalar, vector or 2D matrix")


class SphericalWaveletTransformOperator(ForwardOperator):
    """Identity measurement + spherical wavelet transform (pxmcmc/forward.py:91-123)."""

    def __init__(self, data, sig_d, setting, L, B, J_min, dirs=1, spin=0, nchains=1):
        transform = SphericalWaveletTransform(L, B, J_min, dirs=dirs, spin=spin, nchains=nchains)
        measurement = Identity(len(data), mw_size(L))
        nparams = mw_size(L) if setting == "analysis" else transform.ncoefs
        super().__init__(data, sig_d, setting, transform=transform, measurement=measurement, nparams=nparams)


class PathIntegralOperator(ForwardOperator):
    """Sparse path-integral measurement + spherical wavelet transform (pxmcmc/forward.py:126-162)."""

    def __init__(self, pathmatrix, data, sig_d, setting, L, B, J_min, dirs=1, spin=0, nchains=1):
        transform = SphericalWaveletTransform(L, B, J_min, dirs=dirs, spin=spin, nchains=nchains)
        measurement = PathIntegral(pathmatrix)
        nparams = mw_size(L) if setting == "analysis" else transform.ncoefs
        super().__init__(data, sig_d, setting, transform=transform, measurement=measurement, nparams=nparams)
