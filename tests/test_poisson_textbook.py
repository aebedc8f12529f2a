"""The in-kernel Poisson sampler (csrc/poisson.cuh, CPU replay) against a numpy restatement of
the textbook algorithm on the SAME Philox4x32-10 counters: Hoermann's PTRS exactly as numpy's
legacy generator spells it (squeeze with v_r, exact test with four logarithms and lgamma; the
reference draws with np.random.poisson, ref:510).  The kernel evaluates the two tests in
cheaper forms (no division for v_r; Stirling's series, two logarithms); the variates have to
be the same ones."""
import ctypes

import numpy as np
import pytest

import emul_support
from _poisson_replay import (assert_field, replay_counts, replay_field, textbook_multiplication,
                             textbook_ptrs)

dp = ctypes.POINTER(ctypes.c_double)


@pytest.mark.parametrize('lam', [10.0, 12.5, 17.0, 30.0, 100.0, 1e4, 1.8e7])
def test_sampler_is_textbook_ptrs_on_the_same_counters(lam):
    lib = emul_support.emulator_library()
    lib.cdll.emul_poisson.argtypes = [ctypes.c_double, ctypes.c_uint64, ctypes.c_uint64,
                                      ctypes.c_int, dp]
    n, seed, first = 200000, 0x1234567ABCDEF, 3_000_000_000     # pixel index past 2^31
    got = np.empty(n)
    lib.cdll.emul_poisson(lam, seed, first, n, got.ctypes.data_as(dp))
    want = textbook_ptrs(lam, seed, first + np.arange(n, dtype=np.int64))
    # the two spellings of the tests can only disagree when a uniform falls within rounding of
    # a decision boundary (~1e-13 per sample)
    assert np.array_equal(got, want)


@pytest.mark.parametrize('lam', [0.5, 5.0, 9.9])
def test_small_lambda_sampler_is_the_multiplication_method(lam):
    lib = emul_support.emulator_library()
    lib.cdll.emul_poisson.argtypes = [ctypes.c_double, ctypes.c_uint64, ctypes.c_uint64,
                                      ctypes.c_int, dp]
    n, seed, first = 50000, 987654321, 12345
    got = np.empty(n)
    lib.cdll.emul_poisson(lam, seed, first, n, got.ctypes.data_as(dp))
    want = textbook_multiplication(lam, seed, first + np.arange(n, dtype=np.int64))
    assert np.array_equal(got, want)


def test_field_check_has_teeth():
    """The whole-field comparison the GPU tests make (tests/_poisson_replay.py) fails on one
    pixel off by one count and on a field drawn for another image index."""
    rng = np.random.default_rng(4)
    lam = np.concatenate([np.zeros(300), rng.uniform(0.0, 10.0, 1500), rng.uniform(10.0, 1e4, 1500),
                          rng.uniform(1.9e7, 2.1e7, 300)]).reshape(1, 36, 100)
    seed = 0xC0FFEE
    field = replay_field(lam, seed, 1, np.float32)
    assert_field(field, lam, seed, 1, np.float32)
    for i in (np.flatnonzero(lam == 0)[7], np.flatnonzero((lam > 0) & (lam < 10))[11],
              np.flatnonzero((lam >= 10) & (lam < 1e4))[13]):
        bad = field.copy()
        bad.flat[i] += 1.0
        with pytest.raises(AssertionError, match='pixel %d ' % i):
            assert_field(bad, lam, seed, 1, np.float32)
    with pytest.raises(AssertionError, match='pixels differ'):
        assert_field(field, lam, seed, 0, np.float32)
    # above 2^24 the fp32 field holds even counts only: the replay rounds the same way
    big = field[lam > 2 ** 24]
    assert (big % 2 == 0).all() and not (replay_counts(lam, seed, 1)[lam > 2 ** 24] % 2 == 0).all()


@pytest.mark.parametrize('fast', [1, 0])
@pytest.mark.parametrize('precision', [32, 64])
def test_cpu_replay_noise_field_is_the_textbook_field(precision, fast):
    """create_data's noise field on the CPU replay of the kernels (fast 2160 rows and generic
    rows, both images) is replay_field of its noiseless images, pixel for pixel."""
    from rescan_line_sted_b200 import _lib
    lib = emul_support.emulator_library()
    rng = np.random.default_rng(6)
    ny, nx, seed = 4, 2048, 0x5EED
    psfs = rng.random((2, 3, 9))
    psfs /= psfs.sum(axis=(1, 2), keepdims=True)
    obj = rng.random((1, ny, nx)) * 8.0
    obj[0, :, 100:400] = 0.0            # dark: exact zeros
    obj[0, :, 700:1200] *= 1e3          # PTRS
    obj[0, :, 1500:1600] = 2e7          # fp32 rounds the counts
    h = _lib.DeconvHandle(lib, psfs, (ny, nx), precision=precision)
    h.set_option('fast_path', fast)
    h.create_data(obj, None, seed)
    assert h.info().Lx == 2160
    dtype = np.float32 if precision == 32 else np.float64
    for k in range(2):
        lam = h.get(_lib.NOISELESS, k)
        assert (lam == 0).any() and ((lam > 0) & (lam < 10)).any() and (lam > 2 ** 24).any()
        assert_field(h.get(_lib.NOISY, k), lam, seed, k, dtype)
    h.close()
