"""The host restatement of the library's Philox noise (oracle/philox_ref.py) is itself a sound generator: the GPU tests
compare the device normals with it, so it must not carry a defect the comparison would then accept.  Seeds are fixed,
so every threshold below is deterministic."""
import numpy as np
from scipy import stats

from oracle import philox_ref as P

N_PAIRS = 1 << 20  # 2^21 normals per draw


def _pairs(seed, stream, step):
    return P.philox_normal2(seed, stream, step, np.arange(N_PAIRS, dtype=np.uint64))


def test_normals_are_standard_normal():
    z0, z1 = _pairs(1234, 5, 3)
    z = np.concatenate([z0, z1])
    assert z.size == 1 << 21 and z.dtype == np.float64
    assert stats.kstest(z, "norm").pvalue > 1e-3
    assert abs(z.mean()) < 5 / np.sqrt(z.size)
    assert abs(z.var() - 1) < 5 * np.sqrt(2 / z.size)
    # tails: both Box-Muller outputs reach beyond 4 sigma at the expected rate (6.3e-5 per normal)
    assert 40 < np.count_nonzero(np.abs(z) > 4) < 220


def test_no_correlation_between_halves_streams_and_steps():
    bound = 5 / np.sqrt(N_PAIRS)
    z0, z1 = _pairs(99, 17, 41)
    assert abs(np.corrcoef(z0, z1)[0, 1]) < bound
    assert abs(np.corrcoef(z0 ** 2, z1 ** 2)[0, 1]) < 2 * bound  # Box-Muller halves share the radius only
    a0, _ = _pairs(99, 18, 41)  # adjacent stream
    assert abs(np.corrcoef(z0, a0)[0, 1]) < bound
    s0, _ = _pairs(99, 17, 42)  # adjacent step
    assert abs(np.corrcoef(z0, s0)[0, 1]) < bound
    # adjacent pairs of one stream (the elements 2p and 2p + 2 of a chain)
    assert abs(np.corrcoef(z0[:-1], z0[1:])[0, 1]) < bound


def test_streams_are_distinct_including_wrap_and_wide_counters():
    pairs = np.arange(64, dtype=np.uint64)
    streams = np.concatenate([np.arange(256), [2 ** 32 - 2, 2 ** 32 - 1]]).astype(np.uint64)
    rows = np.stack([np.concatenate(P.philox_normal2(7, s, 1, pairs)) for s in streams])
    assert len({r.tobytes() for r in rows}) == len(streams)
    # the high words of step and seed enter the counter / key: no aliasing with the low words
    base = P.philox_normal2(7, 3, 1, pairs)[0]
    for seed, step in ((7 + 2 ** 32, 1), (7, 1 + 2 ** 32), (2 ** 64 - 1, 2 ** 64 - 1)):
        assert not np.array_equal(P.philox_normal2(seed, 3, step, pairs)[0], base)
    # pair counter above 2^32: the high word is used
    assert not np.array_equal(P.philox_normal2(7, 3, 1, pairs + np.uint64(2 ** 32))[0], base)


def test_uniform_layout_matches_philox_normal2_counter():
    """`philox_uniform` is the first uniform of the counter block (0xFFFFFFFF, 0xFFFFFFFF) -- the block a pair index of
    2^64 - 1 would address -- and lies in (0, 1)"""
    for seed, stream, step in ((77, 2, 1), (2 ** 32 + 5, 2 ** 32 - 1, 2 ** 33 + 7), (0, 0, 0)):
        u1, _ = P.philox_uniforms(seed, stream, step, np.uint64(2 ** 64 - 1))
        u = P.philox_uniform(seed, stream, step)
        assert u == float(u1) and 0.0 < u < 1.0
    # stream ids are 32-bit: stream 2^32 is stream 0
    assert P.philox_uniform(5, 2 ** 32, 9) == P.philox_uniform(5, 0, 9)


def test_element_maps():
    seed, step, s0, nch, n = 11, 6, 2 ** 32 - 3, 4, 7
    w2, z2 = P.element_normals(2, nch, n, seed, step, s0)
    w3r, w3i = P.element_normals(3, nch, n, seed, step, s0)
    w4r, w4i = P.element_normals(4, nch, n, seed, step, s0)
    assert not z2.any()
    for c in range(nch):
        st = (s0 + c) % 2 ** 32
        for e in range(n):
            z0, z1 = P.philox_normal2(seed, st, step, e >> 1)
            assert w2[c, e] == (z1 if e & 1 else z0)
            z0, z1 = P.philox_normal2(seed, st, step, e)
            assert (w3r[c, e], w3i[c, e]) == (z0, z1)
    # packed real chain pairs draw the normals of the unpacked real chains 2c and 2c + 1
    wu, _ = P.element_normals(2, 2 * nch, n, seed, step, s0)
    assert np.array_equal(w4r, wu[0::2]) and np.array_equal(w4i, wu[1::2])
