"""Host restatement of the library's Philox noise (pxmcmc_b200/csrc/pxm_elem.cu).

Every device-noise chain draws its normals from `philox_normal2(seed, stream, step, pair)`: Philox4x32-10 with

    counter = (pair_lo, pair_hi, step_lo, step_hi ^ (stream * 0x85EBCA6B))
    key     = (seed_lo, seed_hi ^ stream)

all words 32-bit.  The four output words make two 64-bit integers a = (w0, w1), b = (w2, w3); their top 53 bits
give the uniforms u = ((x >> 11) + 0.5) 2^-53 in (0, 1), and Box-Muller turns (u1, u2) into

    z0 = sqrt(-2 log u1) cos(2 pi u2),   z1 = sqrt(-2 log u1) sin(2 pi u2).

The uniforms are formed in float64 exactly as the device forms them; the normals are evaluated in np.longdouble and
rounded once, so they are the correctly rounded values to within the extended precision (the device's `log` and
`sincospi` are accurate to a few ulp, not correctly rounded).

Which normal an element uses depends on the kernel (`element_normals`):

* update mode 2 (complex state, real noise; `k_myula_update_pair`) and `k_philox_normal`: element e of chain c is
  normal (e & 1) of pair e >> 1 of stream stream0 + c;
* update mode 3 (complex noise; `k_myula_update`): element e of chain c is (z0, z1) of pair e of stream stream0 + c, as
  (real, imaginary) part;
* update mode 4 (real chain pairs packed into one complex chain; `k_myula_update_realpair`): the real part of element e
  of packed chain c is normal (e & 1) of pair e >> 1 of stream stream0 + 2c, the imaginary part the same of stream
  stream0 + 2c + 1;

with stream ids wrapping modulo 2^32 (`unsigned int` on the device).  The PxMALA accept test draws its uniform from
the counter (0xFFFFFFFF, 0xFFFFFFFF, ...) no coefficient pair reaches (`philox_uniform`).
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
_MUL0, _MUL1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_STREAM_MUL = np.uint64(0x85EBCA6B)
_S32 = np.uint64(32)
# pi to extended precision (np.pi is the float64 value)
_PI_LD = np.longdouble("3.14159265358979323846264338327950288")


def _u64(x):
    return np.asarray(x, dtype=np.uint64) if not isinstance(x, int) else np.uint64(x)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """ten Philox4x32 rounds on uint64 arrays holding 32-bit words (broadcast); returns the four output words"""
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(*(np.asarray(v, dtype=np.uint64) for v in (c0, c1, c2, c3, k0, k1)))
    c0, c1, c2, c3, k0, k1 = (v.copy() for v in (c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0 = _MUL0 * c0
        p1 = _MUL1 * c2
        c0, c1, c2, c3 = ((p1 >> _S32) ^ c1 ^ k0) & M32, p1 & M32, ((p0 >> _S32) ^ c3 ^ k1) & M32, p0 & M32
        k0 = (k0 + _W0) & M32
        k1 = (k1 + _W1) & M32
    return c0, c1, c2, c3


def _keyed_counter(seed, stream, step):
    seed, stream, step = _u64(seed), _u64(stream) & M32, _u64(step)
    c2 = step & M32
    c3 = (step >> _S32) ^ ((stream * _STREAM_MUL) & M32)
    return c2, c3, seed & M32, (seed >> _S32) ^ stream


def _uniform53(hi, lo):
    """((hi:lo) >> 11) + 0.5) * 2^-53 in float64, the device's operation order"""
    bits = (hi << _S32) | lo
    return ((bits >> np.uint64(11)).astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def philox_uniforms(seed, stream, step, pair):
    """(u1, u2) of `philox_normal2` for (seed, stream, step, pair), broadcast over arrays"""
    c2, c3, k0, k1 = _keyed_counter(seed, stream, step)
    pair = _u64(pair)
    w0, w1, w2, w3 = philox4x32_10(pair & M32, pair >> _S32, c2, c3, k0, k1)
    return _uniform53(w0, w1), _uniform53(w2, w3)


def box_muller(u1, u2):
    """(z0, z1) from uniforms in (0, 1), evaluated in np.longdouble and rounded to float64 once"""
    r = np.sqrt(np.longdouble(-2.0) * np.log(np.asarray(u1, dtype=np.longdouble)))
    t = np.asarray(u2, dtype=np.longdouble) * (2 * _PI_LD)
    return (r * np.cos(t)).astype(np.float64), (r * np.sin(t)).astype(np.float64)


def philox_normal2(seed, stream, step, pair):
    """the two standard normals the device draws for (seed, stream, step, pair), broadcast over arrays"""
    return box_muller(*philox_uniforms(seed, stream, step, pair))


def philox_uniform(seed, stream, step):
    """the uniform of the device-resident PxMALA accept test (`k_pxmala_accept`) of chain stream `stream` at `step`"""
    c2, c3, k0, k1 = _keyed_counter(seed, stream, step)
    w0, w1, _, _ = philox4x32_10(M32, M32, c2, c3, k0, k1)
    return float(_uniform53(w0, w1))


def element_normals(mode, nchains, n, seed, step, stream0=0):
    """(w_re, w_im) [nchains, n] float64: the noise every element of the MYULA update draws in Philox `mode`
    (2: real noise, 3: complex noise, 4: packed real chain pairs; `k_philox_normal` is mode 2's w_re)"""
    c = np.arange(nchains, dtype=np.uint64)[:, None]
    e = np.arange(n, dtype=np.uint64)[None, :]
    s0 = np.uint64(stream0)
    one = np.uint64(1)
    if mode == 3:
        return philox_normal2(seed, (s0 + c) & M32, step, e)
    half = (e & one).astype(bool)

    def real_stream(stream):
        z0, z1 = philox_normal2(seed, stream & M32, step, e >> one)
        return np.where(half, z1, z0)

    if mode == 2:
        return real_stream(s0 + c), np.zeros((nchains, n))
    if mode == 4:
        return real_stream(s0 + np.uint64(2) * c), real_stream(s0 + np.uint64(2) * c + one)
    raise ValueError(f"not a Philox update mode: {mode}")
