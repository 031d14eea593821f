"""tests/golden/dsp_golden.npz: what the reference's own STFT / iSTFT / patcher / cross-fade functions computed
(tests/golden/make_golden.py), stored small enough to keep in the repository.

The random inputs are not stored: the functions below regenerate them from integer seeds with integer
arithmetic, so they come out bit for bit the same on every platform and numpy version.  Each output of the
reference is stored as its shape, the SHA-256 of its bytes and its values at a seeded sample of positions;
`check` holds an array to all three, which is as strict as comparing it with the whole stored array."""
import hashlib

import numpy as np

# (frame size, hop, window, samples) of the STFT / iSTFT cases
STFT_CASES = [(1024, 512, "hanning", 5000), (2048, 512, "hanning", 7013), (4096, 512, "blackmanharris", 9001),
              (1024, 256, "sinebell", 3000), (1024, 512, "hanning", 512), (1024, 512, "hanning", 1)]
# (frames, bins, time_context, overlap, batch_size) of the patcher / cross-fade cases
PATCH_CASES = [(100, 17, 30, 25, 32), (64, 9, 30, 20, 8), (30, 5, 30, 25, 32), (31, 5, 30, 25, 4), (203, 7, 20, 15, 16)]
CF_SAMPLES = 6000
PAT3D_SHAPE = (4, 57, 11)
SAMPLE = 64


def uniform(stream, shape):
    """Values in [0, 1), multiples of 2**-53: splitmix64 of (stream, flat index)."""
    n = int(np.prod(shape, dtype=np.int64))
    z = (np.arange(n, dtype=np.uint64) + np.uint64(stream << 40)) * np.uint64(0x9E3779B97F4A7C15)
    z ^= z >> np.uint64(30)
    z *= np.uint64(0xBF58476D1CE4E5B9)
    z ^= z >> np.uint64(27)
    z *= np.uint64(0x94D049BB133111EB)
    z ^= z >> np.uint64(31)
    return ((z >> np.uint64(11)).astype(np.float64) * 2.0 ** -53).reshape(shape)


def signal(stream, n):
    return (uniform(stream, (n,)) - 0.5) * 0.25


def stft_inputs(ci):
    """The signal of STFT case `ci`, and a spectrum of the same shape that is not the STFT of any real
    signal (non-zero imaginary parts at DC and Nyquist exercise irfft's "ignore them")."""
    N, H, _, L = STFT_CASES[ci]
    shape = (-(-L // H) + 2, N // 2 + 1)
    Z = np.empty(shape, dtype=np.complex128)
    Z.real = uniform(1100 + ci, shape) - 0.5
    Z.imag = uniform(1200 + ci, shape) - 0.5
    return signal(1000 + ci, L), Z


def cf_input():
    return signal(1300, CF_SAMPLES)


def patch_input(ci):
    T, F = PATCH_CASES[ci][:2]
    return uniform(1400 + ci, (T, F))


def patch_pred(ci, n):
    """Network outputs [batches, 4 sources, batch_size, 1, time_context, bins] for the n patches of case `ci`."""
    _, F, tc, _, bs = PATCH_CASES[ci]
    return uniform(1500 + ci, (-(-n // bs), 4, bs, 1, tc, F))


def pat3d_input():
    return uniform(1600, PAT3D_SHAPE)


def digest(a):
    """SHA-256 of the little-endian bytes (float64 or complex128; -0.0 counts as 0.0)."""
    a = np.asarray(a)
    dt = "<c16" if np.iscomplexobj(a) else "<f8"
    return hashlib.sha256((np.ascontiguousarray(a, dtype=dt) + 0.0).tobytes()).hexdigest()


def record(key, a, stream):
    """The stored form of output `a`: {key_shape, key_sha256, key_at (sorted flat positions), key_val}."""
    a = np.asarray(a)
    at = np.zeros(0, dtype=np.int64)
    if a.size:
        at = np.unique(np.concatenate([[0, a.size - 1], (uniform(stream, (SAMPLE,)) * a.size).astype(np.int64)]))
    return {key + "_shape": np.array(a.shape, dtype=np.int64), key + "_sha256": np.array(digest(a)),
            key + "_at": at, key + "_val": a.reshape(-1)[at]}


def check(g, key, a):
    """`a` is, bit for bit, the output the reference computed under `key`."""
    a = np.asarray(a)
    assert a.shape == tuple(int(v) for v in g[key + "_shape"]), (key, a.shape)
    assert a.dtype == g[key + "_val"].dtype, (key, a.dtype)
    np.testing.assert_array_equal(a.reshape(-1)[g[key + "_at"]], g[key + "_val"], err_msg=key)
    assert digest(a) == str(g[key + "_sha256"]), "%s differs from the reference away from the sampled positions" % key


def load(path):
    """The stored arrays plus the regenerated inputs under the names the tests use."""
    g = dict(np.load(path))
    for ci in range(len(STFT_CASES)):
        g["stft%d_x" % ci], g["stft%d_Z" % ci] = stft_inputs(ci)
    g["cf_x"] = cf_input()
    for ci in range(len(PATCH_CASES)):
        g["pat%d_m" % ci] = patch_input(ci)
        n = int(g["pat%d_n" % ci])
        if n:
            g["pat%d_pred" % ci] = patch_pred(ci, n)
    g["pat3d_m"] = pat3d_input()
    return g
