"""Device plumbing: torch tensors own the HBM, the C ABI does the arithmetic.

PyTorch is used only for allocation, host<->device copies and the current
stream; every operation on the sampler's hot path is a kernel of
libpxmcmc_b200.so.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, lib, ptr, stream_ptr

CDT = torch.complex128
FDT = torch.float64


def dev():
    _lib.ensure_device()
    return torch.device("cuda", torch.cuda.current_device())


def is_dev(x):
    return isinstance(x, torch.Tensor)


def to_dev_c(x):
    """anything array-like (real or complex) -> contiguous complex128 CUDA tensor"""
    if is_dev(x):
        t = x
        if t.dtype != CDT:
            if t.is_complex():
                t = t.to(CDT)
            else:
                out = torch.empty(t.shape, dtype=CDT, device=t.device)
                tt = t.to(FDT).contiguous()
                check(lib.pxm_real_to_complex(ptr(tt), ptr(out), tt.numel(), stream_ptr()))
                return out
        return t.contiguous()
    a = np.ascontiguousarray(np.asarray(x), dtype=np.complex128)
    if not a.flags.writeable:
        a = a.copy()
    return torch.from_numpy(a).to(dev())


def to_dev_f(x):
    if is_dev(x):
        return x.to(FDT).contiguous()
    a = np.ascontiguousarray(np.asarray(x), dtype=np.float64)
    if not a.flags.writeable:
        a = a.copy()
    return torch.from_numpy(a).to(dev())


def to_host(t):
    return t.detach().cpu().numpy()


def like_input(result, template):
    """numpy in -> numpy out; device tensor in -> device tensor out"""
    return result if is_dev(template) else to_host(result)


# ---------------------------------------------------------------------------
# output placement: a captured iteration must leave its results in the buffers it
# started from (state X, predictions P).  The samplers ask for that with
# `with output_into(buf): ...`; the next result tensor of exactly that shape
# allocated through `new_c` below IS `buf` (no copy kernel, no ATen op).  Callers
# check the returned tensor and fall back to `copy_into` when an operator they do
# not know allocated its result some other way.
# ---------------------------------------------------------------------------
_out_hint = [None]


class output_into:
    def __init__(self, buf):
        self.buf = buf

    def __enter__(self):
        self.prev = _out_hint[0]
        _out_hint[0] = self.buf
        return self

    def __exit__(self, *exc):
        _out_hint[0] = self.prev
        return False


def new_c(shape, device):
    """uninitialised complex128 result tensor (or the pending `output_into` buffer of that shape)"""
    h = _out_hint[0]
    if h is not None and tuple(h.shape) == tuple(shape) and h.device == device:
        _out_hint[0] = None
        return h
    return torch.empty(tuple(shape), dtype=CDT, device=device)


def copy_into(dst, src):
    """dst <- src (complex128, same shape) with the library's own kernel; no-op when they are the same buffer"""
    if dst.data_ptr() == src.data_ptr():
        return dst
    arr = (C.c_void_p * 4)(src.data_ptr(), 0, 0, 0)
    cf = (C.c_double * 4)(1.0, 0.0, 0.0, 0.0)
    check(lib.pxm_lincomb(1, arr, cf, None, 0.0, 0.0, ptr(dst), dst.numel(), stream_ptr()))
    return dst


def batch2d(t):
    """view a [n] or [nb, n] tensor as ([nb, n], was_1d)"""
    if t.dim() == 1:
        return t.unsqueeze(0), True
    if t.dim() == 2:
        return t, False
    raise ValueError("expected a 1-D vector or a [nchains, n] batch")


# ---------------------------------------------------------------------------
# plans
# ---------------------------------------------------------------------------
class WaveletPlan:
    """pxm_wav_plan: all four wavelet operators for one (L, B, J_min, nbatch)."""

    _cache = {}

    @classmethod
    def get(cls, L, B, J_min, nbatch):
        key = (int(L), float(B), int(J_min), int(nbatch), torch.cuda.current_device() if torch.cuda.is_available() else -1)
        if key not in cls._cache:
            cls._cache[key] = cls(L, B, J_min, nbatch)
        return cls._cache[key]

    def __init__(self, L, B, J_min, nbatch):
        dev()
        self.L, self.B, self.J_min, self.nbatch = int(L), float(B), int(J_min), int(nbatch)
        h = C.c_void_p()
        check(lib.pxm_wav_plan_create(self.L, self.B, self.J_min, self.nbatch, C.byref(h)))
        self.h = h
        ns, nc, nsc, J, tb = C.c_int(), C.c_longlong(), C.c_longlong(), C.c_int(), C.c_longlong()
        check(lib.pxm_wav_plan_info(h, C.byref(ns), C.byref(nc), C.byref(nsc), C.byref(J), C.byref(tb)))
        self.nscales_total, self.ncoefs, self.nscal, self.J_max, self.table_bytes = ns.value, nc.value, nsc.value, J.value, tb.value
        bl = (C.c_int * ns.value)()
        check(lib.pxm_wav_plan_bandlimits(h, bl, ns.value))
        self.bandlimits = list(bl)
        self.npix = self.L * (2 * self.L - 1)

    def _run(self, fn, x, n_in, n_out, in_first):
        x2, was1 = batch2d(x)
        nb = x2.shape[0]
        if x2.shape[1] != n_in:
            raise ValueError(f"expected vectors of length {n_in}, got {x2.shape[1]}")
        if nb > self.nbatch:
            raise ValueError("batch larger than the plan's")
        out = new_c((nb, n_out), x2.device)
        check(fn(self.h, ptr(x2), ptr(out), nb, stream_ptr()))
        return out[0] if was1 else out

    def synthesis(self, coef):
        return self._run(lib.pxm_wav_synthesis, coef, self.ncoefs, self.npix, True)

    def synthesis_adjoint(self, pix):
        return self._run(lib.pxm_wav_synthesis_adjoint, pix, self.npix, self.ncoefs, True)

    def analysis(self, pix):
        return self._run(lib.pxm_wav_analysis, pix, self.npix, self.ncoefs, True)

    def analysis_adjoint(self, coef):
        return self._run(lib.pxm_wav_analysis_adjoint, coef, self.ncoefs, self.npix, True)

    def synthesis_harmonic(self, coef):
        """synthesis stopped in harmonic space: coefficients -> f_lm [L^2] of the image"""
        return self._run(lib.pxm_wav_synthesis_harmonic, coef, self.ncoefs, self.L * self.L, True)

    def synthesis_adjoint_harmonic(self, flm):
        """adjoint of `synthesis_harmonic`"""
        return self._run(lib.pxm_wav_synthesis_adjoint_harmonic, flm, self.L * self.L, self.ncoefs, True)


    # ---- ring-Fourier form of the pixel side (pxm_wav_*_ring*): float64 tensors [ring_doubles] in the plan's layout
    @property
    def ring_doubles(self):
        return int(lib.pxm_wav_ring_doubles(self.h))

    def new_ring(self, device, like=None):
        if like is not None:
            return like
        return torch.empty(self.ring_doubles, dtype=FDT, device=device)

    def synthesis_to_ring(self, coef, out=None):
        c2, _ = batch2d(coef)
        if c2.shape[1] != self.ncoefs or c2.shape[0] > self.nbatch:
            raise ValueError("coefficient batch does not fit the plan")
        ring = self.new_ring(c2.device, out)
        check(lib.pxm_wav_synthesis_to_ring(self.h, ptr(c2), ptr(ring), c2.shape[0], stream_ptr()))
        return ring

    def synthesis_adjoint_from_ring(self, ring, nb):
        out = torch.empty((nb, self.ncoefs), dtype=CDT, device=ring.device)
        check(lib.pxm_wav_synthesis_adjoint_from_ring(self.h, ptr(ring), ptr(out), nb, stream_ptr()))
        return out

    def ring_to_pix(self, ring, nb):
        out = torch.empty((nb, self.npix), dtype=CDT, device=ring.device)
        check(lib.pxm_wav_ring_to_pix(self.h, ptr(ring), ptr(out), nb, stream_ptr()))
        return out

    def pix_to_ring(self, pix, out=None):
        p2, _ = batch2d(pix)
        if p2.shape[1] != self.npix or p2.shape[0] > self.nbatch:
            raise ValueError("pixel batch does not fit the plan")
        ring = out if out is not None else torch.zeros(self.ring_doubles, dtype=FDT, device=p2.device)
        check(lib.pxm_wav_pix_to_ring(self.h, ptr(p2), ptr(ring), p2.shape[0], stream_ptr()))
        return ring

    def ring_resid(self, pred, data_ring, ic_rings, nb, out=None):
        """ic[t] * ((2L-1) pred - data) on ring arrays; ic_rings: complex128 [L]"""
        ring = self.new_ring(pred.device, out)
        check(lib.pxm_wav_ring_resid(self.h, ptr(pred), ptr(data_ring), ptr(ic_rings), ptr(ring), nb, stream_ptr()))
        return ring


    # ---- harmonic (Gram) form of the pixel side (pxm_wav_*harm*, pxm_wav_gram_gradient): float64 tensors [harm_doubles]
    @property
    def harm_doubles(self):
        return int(lib.pxm_wav_harm_doubles(self.h))

    def synthesis_to_harm(self, coef, out=None):
        c2, _ = batch2d(coef)
        if c2.shape[1] != self.ncoefs or c2.shape[0] > self.nbatch:
            raise ValueError("coefficient batch does not fit the plan")
        # (the contraction writes every row of every slot, padding included: no initialisation needed)
        harm = out if out is not None else torch.empty(self.harm_doubles, dtype=FDT, device=c2.device)
        check(lib.pxm_wav_synthesis_to_harm(self.h, ptr(c2), ptr(harm), c2.shape[0], stream_ptr()))
        return harm

    def set_gram_weights(self, w, key=None):
        """per-ring weights of the Gram table (None: all one); `key` identifies them so that callers can tell whether the
        table still is theirs (`gram_key`)"""
        import ctypes as C

        if w is None:
            check(lib.pxm_wav_set_gram_weights(self.h, None, 0))
        else:
            w = np.ascontiguousarray(w, dtype=np.float64)
            check(lib.pxm_wav_set_gram_weights(self.h, w.ctypes.data_as(C.POINTER(C.c_double)), int(w.size)))
        self.gram_key = key

    gram_key = None

    def gram_gradient(self, harm, b_harm, ic, nb):
        out = torch.empty((nb, self.ncoefs), dtype=CDT, device=harm.device)
        check(lib.pxm_wav_gram_gradient(self.h, ptr(harm), ptr(b_harm), float(ic.real), float(ic.imag), ptr(out), nb, stream_ptr()))
        return out

    def harm_to_pix(self, harm, nb):
        out = torch.empty((nb, self.npix), dtype=CDT, device=harm.device)
        check(lib.pxm_wav_harm_to_pix(self.h, ptr(harm), ptr(out), nb, stream_ptr()))
        return out

    def pix_to_harm_adjoint(self, pix):
        p2, _ = batch2d(pix)
        harm = torch.zeros(self.harm_doubles, dtype=FDT, device=p2.device)
        check(lib.pxm_wav_pix_to_harm_adjoint(self.h, ptr(p2), ptr(harm), p2.shape[0], stream_ptr()))
        return harm


class ShtPlan:
    """pxm_sht_plan: the four pyssht-level transforms for one (L, spin, nbatch)."""

    _cache = {}

    @classmethod
    def get(cls, L, spin, nbatch=1):
        key = (int(L), int(spin), int(nbatch), torch.cuda.current_device() if torch.cuda.is_available() else -1)
        if key not in cls._cache:
            cls._cache[key] = cls(L, spin, nbatch)
        return cls._cache[key]

    def __init__(self, L, spin, nbatch=1):
        dev()
        self.L, self.spin, self.nbatch = int(L), int(spin), int(nbatch)
        h = C.c_void_p()
        check(lib.pxm_sht_plan_create(self.L, self.spin, self.nbatch, C.byref(h)))
        self.h = h
        self.npix = self.L * (2 * self.L - 1)
        self.nlm = self.L * self.L

    def _run(self, fn, x, n_in, n_out, gl):
        x2, was1 = batch2d(x)
        nb = x2.shape[0]
        if x2.shape[1] != n_in:
            raise ValueError(f"expected vectors of length {n_in}, got {x2.shape[1]}")
        out = new_c((nb, n_out), x2.device)
        check(fn(self.h, ptr(x2), ptr(out), nb, ptr(gl), stream_ptr()))
        return out[0] if was1 else out

    # argument order of the C ABI is (in, out) for every call
    def inverse(self, flm, gl=None):
        return self._run(lib.pxm_sht_inverse, flm, self.nlm, self.npix, gl)

    def forward(self, f, gl=None):
        return self._run(lib.pxm_sht_forward, f, self.npix, self.nlm, gl)

    def inverse_adjoint(self, f, gl=None):
        return self._run(lib.pxm_sht_inverse_adjoint, f, self.npix, self.nlm, gl)

    def forward_adjoint(self, flm, gl=None):
        return self._run(lib.pxm_sht_forward_adjoint, flm, self.nlm, self.npix, gl)


# ---------------------------------------------------------------------------
# elementwise wrappers (device tensors in / out)
# ---------------------------------------------------------------------------
def _T_args(T):
    """threshold as (device vector or None, scalar)"""
    if is_dev(T):
        return T, 0.0
    if np.ndim(T) == 0:
        return None, float(T)
    return to_dev_f(T), 0.0


def soft_dev(x, Tvec, Tscalar):
    x2, was1 = batch2d(x)
    out = torch.empty_like(x2)
    n = x2.shape[1]
    if Tvec is not None and Tvec.numel() != n:
        raise ValueError("threshold vector has the wrong length")
    check(lib.pxm_soft(1 if x2.is_complex() else 0, ptr(x2), ptr(Tvec), Tscalar, ptr(out), n, x2.shape[0], stream_ptr()))
    return out[0] if was1 else out


def myula_update_dev(X, prox, gradg, Tvec, Tscalar, delta, lmda, w_re=None, w_im=None, noise_mode=0, seed=0, step=0,
                     stream0=0, want_prox=False, dstep=None, out=None):
    """dstep: int64 device tensor holding the Philox step (read by the kernel, then advanced by one):
    the form a captured CUDA graph can replay.  `out` may be X itself (every thread reads its elements before it
    writes them)."""
    X2, was1 = batch2d(X)
    nb, n = X2.shape
    out = torch.empty_like(X2) if out is None else batch2d(out)[0]
    pout = torch.empty_like(X2) if want_prox else None
    if dstep is not None:
        check(lib.pxm_myula_update_dstep(ptr(X2), ptr(prox), ptr(gradg), ptr(Tvec), Tscalar, ptr(out), ptr(pout), n, nb,
                                         float(delta), float(lmda), int(noise_mode), int(seed), ptr(dstep), int(stream0),
                                         stream_ptr()))
        check(lib.pxm_counter_add(ptr(dstep), 1, stream_ptr()))
    else:
        check(lib.pxm_myula_update(ptr(X2), ptr(prox), ptr(gradg), ptr(Tvec), Tscalar, ptr(w_re), ptr(w_im), ptr(out),
                                   ptr(pout), n, nb, float(delta), float(lmda), int(noise_mode), int(seed), int(step),
                                   int(stream0), stream_ptr()))
    if was1:
        out = out[0]
        pout = pout[0] if pout is not None else None
    return (out, pout) if want_prox else out


_scratch = {}


def myula_update_dpar_dev(X, prox, gradg, Tvec, Tscalar, dpar, noise_mode, seed, step, stream0=0):
    """the proposal with {delta, 1-delta/lmda, delta/lmda, sqrt(2 delta)} read from the device block `dpar`"""
    X2, was1 = batch2d(X)
    nb, n = X2.shape
    out = torch.empty_like(X2)
    check(lib.pxm_myula_update_dpar(ptr(X2), ptr(prox), ptr(gradg), ptr(Tvec), Tscalar, ptr(out), None, n, nb, ptr(dpar),
                                    int(noise_mode), int(seed), int(step), int(stream0), stream_ptr()))
    return out[0] if was1 else out


def reduce_dpar_dev(a, b, c, d, dpar, lmda):
    """kind-2 reduction (PxMALA transition) with the step size read from the device block `dpar`"""
    a2, _ = batch2d(a)
    nb, n = a2.shape
    key = (nb, a2.device, torch.cuda.current_stream().cuda_stream)  # concurrent reductions on different streams do not share scratch
    if key not in _scratch:
        _scratch[key] = torch.empty(nb * lib.pxm_reduce_scratch_elems(), dtype=CDT, device=a2.device)
    out = torch.empty(nb, dtype=CDT, device=a2.device)
    check(lib.pxm_reduce_dpar(2, ptr(a2), ptr(b), ptr(c), ptr(d), None, ptr(dpar), float(lmda), n, nb, ptr(_scratch[key]),
                              ptr(out), stream_ptr()))
    return out


def pxmala_accept_dev(state, s1, s2, L2p, priorp, mu, lmda, tune, i, seed, step, stream_id, acc_trace, delta_trace):
    """state [nchains, 16]; acc_trace int8 [nchains, cap]; delta_trace float64 [nchains, cap + 1]"""
    nch, cap = acc_trace.shape
    check(lib.pxm_pxmala_accept(ptr(state), ptr(s1), ptr(s2), ptr(L2p), ptr(priorp), float(mu), float(lmda), int(bool(tune)),
                                int(i), int(seed), int(step), int(stream_id), ptr(acc_trace), ptr(delta_trace), cap, nch,
                                stream_ptr()))


def select_if_dev(state, dsts, srcs):
    """dst_k[c] <- src_k[c] ([nchains, n_k] complex tensors) for the chains whose state block says `accepted`"""
    k = len(dsts)
    nch = state.shape[0]
    d = (C.c_void_p * 4)(*([t.data_ptr() for t in dsts] + [0] * (4 - k)))
    sr = (C.c_void_p * 4)(*([t.data_ptr() for t in srcs] + [0] * (4 - k)))
    cnt = (C.c_longlong * 4)(*([t.numel() // nch for t in dsts] + [0] * (4 - k)))
    check(lib.pxm_select_if(C.c_void_p(state.data_ptr() + 9 * 8), state.shape[1], nch, d, sr, cnt, k, stream_ptr()))


def philox_normal_dev(nchains, n, seed, step=0, stream0=0, dstep=None):
    """[nchains, n] float64 standard normals from the library's Philox streams (step from `dstep` when given)"""
    out = torch.empty((nchains, n), dtype=FDT, device=dev())
    check(lib.pxm_philox_normal(ptr(out), n, nchains, int(seed), int(step), ptr(dstep), int(stream0), stream_ptr()))
    return out


def gradlogpi_dev(X, prox, Tvec, Tscalar, gradg, lmda):
    X2, was1 = batch2d(X)
    out = torch.empty_like(X2)
    check(lib.pxm_gradlogpi(ptr(X2), ptr(prox), ptr(Tvec), Tscalar, ptr(gradg), float(lmda), ptr(out), X2.shape[1],
                            X2.shape[0], stream_ptr()))
    return out[0] if was1 else out


class SkrockNoise:
    """the Z of one SKROCK step for pxm_skrock_shift / pxm_skrock_stage: injected real normals `re` [nchains, n] (and
    `im` for complex chains), or, with re = None, the Philox normals pxm_philox_normal draws at (seed, stream0 + chain,
    step) -- step read from the int64 device tensor `dstep` when given -- real or (`complex`) one 2n draw per chain"""

    def __init__(self, re=None, im=None, *, complex=False, seed=0, step=0, stream0=0, dstep=None):
        self.re, self.im = (None if re is None else to_dev_f(re)), (None if im is None else to_dev_f(im))
        if self.re is None:
            self.mode = 4 if complex else 3
        else:
            self.mode = 2 if self.im is not None else 1
        self.seed, self.step, self.stream0, self.dstep = int(seed), int(step), int(stream0), dstep

    def args(self):
        return (ptr(self.re), ptr(self.im), self.mode, self.seed, self.step, ptr(self.dstep), self.stream0)


def skrock_shift_dev(X, c, Z, out=None):
    """Y = X + c Z ([nchains, n] complex; Z a `SkrockNoise`)"""
    X2, was1 = batch2d(X)
    out = torch.empty_like(X2) if out is None else batch2d(out)[0]
    check(lib.pxm_skrock_shift(ptr(X2), float(c), *Z.args(), ptr(out), X2.shape[1], X2.shape[0], stream_ptr()))
    return out[0] if was1 else out


def skrock_stage_dev(U, V, gradg, prox, Tvec, Tscalar, lmda, a, b, c, c0, Z=None, c_shift=0.0, e=0.0, out=None):
    """one SKROCK stage: a g + b U + c V + c0 (+ e Z), g = grad log pi at P = U (+ c_shift Z); see pxm_skrock_stage.
    V = None is stage 1.  `out` may be U or V."""
    U2, was1 = batch2d(U)
    out = torch.empty_like(U2) if out is None else batch2d(out)[0]
    zargs = Z.args() if Z is not None else (None, None, 0, 0, 0, None, 0)
    check(lib.pxm_skrock_stage(ptr(U2), ptr(V), ptr(gradg), ptr(prox), ptr(Tvec), float(Tscalar), float(lmda), float(a),
                               float(b), float(c), float(c0), float(c_shift), float(e), *zargs, ptr(out), U2.shape[1],
                               U2.shape[0], stream_ptr()))
    return out[0] if was1 else out


def fista_update_dev(Y, gradg, X, Tvec, Tscalar, Tscale, t, state, hist, out=None):
    """one FISTA iteration (pxm_fista_update) of the [nchains, n] complex tensors: (x_{k+1}, y_{k+1}) written to `out`
    (X, Y themselves are allowed) or to new tensors; `state` = float64 device tensor {k, tau_k}, advanced by the call;
    `hist` = float64 [cap, nchains, 2] receives |x_{k+1} - x_k|^2 and |x_{k+1}|^2 in slot k mod cap"""
    nb, n = Y.shape
    if hist.dim() != 3 or hist.shape[1:] != (nb, 2) or hist.dtype != FDT:
        raise ValueError("fista_update: hist must be a float64 [cap, nchains, 2] tensor")
    Xo, Yo = (torch.empty_like(Y), torch.empty_like(Y)) if out is None else out
    key = (nb, Y.device, torch.cuda.current_stream().cuda_stream)
    if key not in _scratch:
        _scratch[key] = torch.empty(nb * lib.pxm_reduce_scratch_elems(), dtype=CDT, device=Y.device)
    check(lib.pxm_fista_update(ptr(Y), ptr(gradg), ptr(X), ptr(Tvec), float(Tscalar), float(Tscale), float(t), ptr(state),
                               ptr(Xo), ptr(Yo), ptr(hist), hist.shape[0], n, nb, ptr(_scratch[key]), stream_ptr()))
    return Xo, Yo


def resid_dev(preds, data, invcov):
    p2, was1 = batch2d(preds)
    out = torch.empty_like(p2)
    check(lib.pxm_resid_invcov(ptr(p2), ptr(data), ptr(invcov), ptr(out), p2.shape[1], p2.shape[0], stream_ptr()))
    return out[0] if was1 else out


def reduce_dev(kind, a, b=None, c=None, d=None, w=None, delta=0.0, lmda=1.0):
    """per-chain complex reductions; returns a [nchains] complex128 device tensor"""
    a2, _ = batch2d(a)
    nb, n = a2.shape
    key = (nb, a2.device, torch.cuda.current_stream().cuda_stream)  # concurrent reductions on different streams do not share scratch
    if key not in _scratch:
        _scratch[key] = torch.empty(nb * lib.pxm_reduce_scratch_elems(), dtype=CDT, device=a2.device)
    out = torch.empty(nb, dtype=CDT, device=a2.device)
    check(lib.pxm_reduce(kind, ptr(a2), ptr(b), ptr(c), ptr(d), ptr(w), float(delta), float(lmda), n, nb,
                         ptr(_scratch[key]), ptr(out), stream_ptr()))
    return out


def lincomb_dev(terms, z=None, cz=0.0, c0=0.0, out=None):
    """sum_k coef_k * x_k (+ cz*z real, + c0 real), complex128 device tensors of equal shape; `out` may alias a term"""
    xs = [t for _, t in terms]
    n = len(xs)
    arr = (C.c_void_p * 4)(*([x.data_ptr() for x in xs] + [0] * (4 - n)))
    cf = (C.c_double * 4)(*([float(c) for c, _ in terms] + [0.0] * (4 - n)))
    if out is None:
        out = torch.empty_like(xs[0])
    check(lib.pxm_lincomb(n, arr, cf, ptr(z), float(cz), float(c0), ptr(out), out.numel(), stream_ptr()))
    return out


def gather_dev(full, idx, w, nsel):
    f2, was1 = batch2d(full)
    out = new_c((f2.shape[0], nsel), f2.device)
    check(lib.pxm_masked_gather(ptr(f2), ptr(idx), ptr(w), ptr(out), nsel, f2.shape[1], f2.shape[0], stream_ptr()))
    return out[0] if was1 else out


def scatter_dev(sel, idx, w, nfull):
    s2, was1 = batch2d(sel)
    out = torch.empty((s2.shape[0], nfull), dtype=CDT, device=s2.device)
    check(lib.pxm_masked_scatter(ptr(s2), ptr(idx), ptr(w), ptr(out), s2.shape[1], nfull, s2.shape[0], stream_ptr()))
    return out[0] if was1 else out


def csr_spmv_dev(indptr, indices, vals, x, nrows, ncols):
    x2, was1 = batch2d(x)
    if x2.shape[1] != ncols:
        raise ValueError("vector length does not match the matrix")
    out = new_c((x2.shape[0], nrows), x2.device)
    check(lib.pxm_csr_spmv(ptr(indptr), ptr(indices), ptr(vals), ptr(x2), ptr(out), nrows, ncols, x2.shape[0], stream_ptr()))
    return out[0] if was1 else out


# ---------------------------------------------------------------------------
# streaming posterior summaries (pxm_stats_*): accumulators are flat float64 tensors in the library's layout
# ---------------------------------------------------------------------------
def stats_accumulator(n, nchains, mode):
    """zeroed accumulator for `nchains` complex chains of length `n` (mode 0 real part, 1 re + im, 2 packed pairs)"""
    nd = int(lib.pxm_stats_accumulator_doubles(int(n), int(nchains), int(mode)))
    if nd < 0:
        raise _lib.PxmError(lib.pxm_last_error().decode())
    acc = torch.empty(nd, dtype=FDT, device=dev())
    check(lib.pxm_stats_reset(ptr(acc), int(n), int(nchains), int(mode), stream_ptr()))
    return acc


def stats_accumulate_dev(acc, x, mode, nsamples, j=0, d_j=None):
    """push sample j (or, per chain, d_j[c]; < 0 skips the chain) of the complex chains x [nchains, n]"""
    x2, _ = batch2d(x)
    if x2.dtype != CDT or not x2.is_contiguous():
        raise ValueError("stats_accumulate: x must be a contiguous complex128 [nchains, n] tensor")
    if d_j is not None and (d_j.dtype != torch.int64 or d_j.numel() != x2.shape[0]):
        raise ValueError("stats_accumulate: d_j must be an int64 tensor with one entry per chain")
    check(lib.pxm_stats_accumulate(ptr(acc), ptr(x2), x2.shape[1], x2.shape[0], int(mode), int(nsamples), int(j), ptr(d_j),
                                   stream_ptr()))


def stats_partials_dev(acc, n, nchains, mode, nsamples, per_chain=True):
    """(record [10, ncomp, n], chain mean [nslots, n] or None, chain variance [nslots, n] or None) device tensors"""
    ncomp = 2 if mode == 1 else 1
    nslots = nchains if mode == 0 else 2 * nchains
    rec = torch.empty((10, ncomp, n), dtype=FDT, device=acc.device)
    cm = torch.empty((nslots, n), dtype=FDT, device=acc.device) if per_chain else None
    cv = torch.empty((nslots, n), dtype=FDT, device=acc.device) if per_chain else None
    check(lib.pxm_stats_partials(ptr(acc), int(n), int(nchains), int(mode), int(nsamples), ptr(rec), ptr(cm), ptr(cv),
                                 stream_ptr()))
    return rec, cm, cv


def rank_diagnostics_dev(x, m, n):
    """(rhat, ess_bulk, ess_tail) [ncols] device tensors of the columns of x, a float64 CUDA tensor [m n, ncols] with
    unit column stride whose row c n + i is sample i of chain c (pxm_rank_diagnostics)"""
    if x.dtype != FDT or x.dim() != 2 or x.shape[0] != m * n or (x.shape[1] > 1 and x.stride(1) != 1):
        raise ValueError("rank_diagnostics: x must be a float64 [m n, ncols] tensor with unit column stride")
    ncols = x.shape[1]
    nd = int(lib.pxm_rank_diagnostics_scratch_doubles(int(m), int(n), ncols))
    if nd < 0:
        raise _lib.PxmError(lib.pxm_last_error().decode())
    scratch = torch.empty(nd, dtype=FDT, device=x.device)
    out = torch.empty((3, ncols), dtype=FDT, device=x.device)
    check(lib.pxm_rank_diagnostics(ptr(x), int(m), int(n), ncols, max(x.stride(0), 1), ptr(scratch), ptr(out[0]),
                                   ptr(out[1]), ptr(out[2]), stream_ptr()))
    return out[0], out[1], out[2]


# ---------------------------------------------------------------------------
# streaming credible intervals (pxm_credible_*): tail heaps in a flat float64 tensor in the library's layout; `tails`
# = (npooled, lo_a, gamma_a, lo_b, gamma_b) as diagnostics.credible_tails gives them
# ---------------------------------------------------------------------------
def credible_state_doubles(n, mode, tails):
    N, lo_a, _, lo_b, _ = tails
    nd = int(lib.pxm_credible_state_doubles(int(n), int(mode), int(N), int(lo_a), int(lo_b)))
    if nd < 0:
        raise _lib.PxmError(lib.pxm_last_error().decode())
    return nd


def credible_state(n, mode, tails):
    """zeroed tail heaps of `n` elements (mode 0 real part, 1 re + im, 2 packed pairs)"""
    N, lo_a, _, lo_b, _ = tails
    st = torch.empty(credible_state_doubles(n, mode, tails), dtype=FDT, device=dev())
    check(lib.pxm_credible_reset(ptr(st), int(n), int(mode), int(N), int(lo_a), int(lo_b), stream_ptr()))
    return st


def credible_push_dev(st, x, mode, tails, count, d_j=None):
    """offer one sample of every chain of x [nchains, n] (with d_j: of the chains whose entry is >= 0); `count`
    samples are pooled per column before this push"""
    x2, _ = batch2d(x)
    if x2.dtype != CDT or not x2.is_contiguous():
        raise ValueError("credible_push: x must be a contiguous complex128 [nchains, n] tensor")
    if d_j is not None and (d_j.dtype != torch.int64 or d_j.numel() != x2.shape[0]):
        raise ValueError("credible_push: d_j must be an int64 tensor with one entry per chain")
    N, lo_a, _, lo_b, _ = tails
    check(lib.pxm_credible_push(ptr(st), ptr(x2), x2.shape[1], x2.shape[0], int(mode), int(N), int(lo_a), int(lo_b),
                                int(count), ptr(d_j), stream_ptr()))


def credible_finalize_dev(st, n, mode, tails):
    """(lower, upper) device tensors [ncomp, n] (ncomp = 2 in mode 1, else 1)"""
    N, lo_a, g_a, lo_b, g_b = tails
    out = torch.empty((2, 2 if mode == 1 else 1, int(n)), dtype=FDT, device=st.device)
    check(lib.pxm_credible_finalize(ptr(st), int(n), int(mode), int(N), int(lo_a), float(g_a), int(lo_b), float(g_b),
                                    ptr(out[0]), ptr(out[1]), stream_ptr()))
    return out[0], out[1]
