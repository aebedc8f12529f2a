"""Overlap-save tiling (objects larger than one shared-memory transform) on the
CPU replay of the kernel bodies: the tiled operators must equal the untiled
ones and the oracle, including the Poisson field."""
import numpy as np
import pytest

import emul_support
from oracle import line_sted_oracle as orc
from rescan_line_sted_b200 import _lib


def rel_l2(a, b):
    return np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b))


@pytest.fixture(scope='module')
def lib():
    return emul_support.emulator_library()


# (shape, PSF shape, tile FFT length).  The first four keep their original ids.
TILED_CASES = [
    pytest.param((150, 170), (9, 11), 64, id='shape0'),
    pytest.param((64, 64), (9, 11), 64, id='shape1'),
    pytest.param((47, 201), (9, 11), 64, id='shape2'),
    pytest.param((57, 56), (9, 11), 64, id='shape3'),
    # even and rectangular PSFs: asymmetric halos (first interior row ny-1-sy != sy)
    pytest.param((150, 170), (10, 12), 64, id='psf10x12'),
    pytest.param((100, 150), (9, 31), 64, id='psf9x31'),
    # 1 x 1 PSF: no halo, the whole window is interior
    pytest.param((150, 170), (1, 1), 64, id='psf1x1'),
    # 1 x N and N x 1 tile grids; last tile row and column one pixel wide (2 * 56 + 1, 2 * 54 + 1)
    pytest.param((40, 200), (9, 11), 64, id='grid1xN'),
    pytest.param((200, 40), (9, 11), 64, id='gridNx1'),
    pytest.param((113, 109), (9, 11), 64, id='last_tile_one_pixel'),
    # other window lengths: radix schedules 16 * 3 and 8 * 9
    pytest.param((100, 90), (9, 11), 48, id='w48'),
    pytest.param((150, 130), (10, 12), 72, id='w72_psf10x12'),
]


@pytest.mark.parametrize('shape,psf_shape,tile_len', TILED_CASES)
@pytest.mark.parametrize('precision,tol', [(64, 1e-12), (32, 1e-5)])
def test_tiled_equals_untiled_and_oracle(lib, shape, psf_shape, tile_len, precision, tol):
    rng = np.random.default_rng(0)
    psfs = rng.random((3,) + psf_shape)
    x = rng.random((1,) + shape)
    y = rng.random((3,) + shape)
    o = orc.Deconvolver([p[None] for p in psfs])
    tiled = _lib.DeconvHandle(lib, psfs, shape, precision=precision, tile_fft_len=tile_len)
    info = tiled.info()
    out_y, out_x = tile_len - (psf_shape[0] - 1), tile_len - (psf_shape[1] - 1)
    assert (info.Ly, info.Lx) == (tile_len, tile_len)
    assert info.tile_out_y == out_y and info.tile_out_x == out_x
    assert info.tiles_y == -(-shape[0] // out_y) and info.tiles_x == -(-shape[1] // out_x)
    assert rel_l2(tiled.H(x), np.concatenate(o.H(x))) < tol
    ylist = [v[None] for v in y]
    assert rel_l2(tiled.Ht(y, False), o.H_t(ylist, normalize=False)) < tol
    assert rel_l2(tiled.Ht(y, True), o.H_t(ylist)) < tol
    plain = _lib.DeconvHandle(lib, psfs, shape, precision=precision)
    assert plain.info().tiles_y == 1
    tiled.create_data(x, 1e7, 5)
    plain.create_data(x, 1e7, 5)
    if precision == 64:  # same Philox counters (global pixel index), same lambda
        for k in range(3):
            assert np.array_equal(tiled.get(_lib.NOISY, k), plain.get(_lib.NOISY, k))
    for k in range(3):
        tiled.set(_lib.NOISY, k, plain.get(_lib.NOISY, k))
    tiled.iterate(3)
    plain.iterate(3)
    assert rel_l2(tiled.get(_lib.ESTIMATE), plain.get(_lib.ESTIMATE)) < 10 * tol
    assert tiled.info().iterations_done == 3
    # record_iteration's error spectrum of a tiled object (direct transform, ref:539-546)
    est, true = tiled.get(_lib.ESTIMATE), tiled.get(_lib.TRUE_OBJECT)
    want = np.log(1 + np.abs(np.fft.fftshift(np.fft.fftn(est - true, axes=(1, 2)), axes=(1, 2))))
    ft_tol = 1e-12 if precision == 64 else 2e-4
    assert np.abs(tiled.ft_error() - want).max() <= ft_tol * np.abs(want).max()
    assert np.abs(tiled.ft_error(est) - want).max() <= ft_tol * np.abs(want).max()
    tiled.close(), plain.close()


def test_tile_shorter_than_psf_is_an_error(lib):
    with pytest.raises(RuntimeError, match='(?i)shorter|too short'):
        _lib.DeconvHandle(lib, np.ones((1, 9, 9)), (40, 40), precision=64, tile_fft_len=8)


def test_tile_length_without_fft_plan_is_an_error(lib):
    """2002 = 2 * 7 * 11 * 13 has no radix schedule: the handle is refused, nothing runs."""
    with pytest.raises(RuntimeError, match='no FFT plan'):
        _lib.DeconvHandle(lib, np.ones((1, 9, 9)), (4000, 4000), precision=32, tile_fft_len=2002)


def test_simulate_uses_the_uploaded_object(lib):
    """A frame loop uploads the object once and simulates per frame; reads, writes and the error
    spectrum in between must not change what simulate() draws from."""
    rng = np.random.default_rng(2)
    psfs = rng.random((2, 9, 11))
    x = rng.random((1, 100, 120)) + 0.1
    want = np.concatenate(orc.Deconvolver([p[None] for p in psfs]).H(x * (1e6 / x.sum())))
    h = _lib.DeconvHandle(lib, psfs, x.shape[1:], precision=64, tile_fft_len=64)
    h.upload_object(x)
    for _ in range(2):
        h.get(_lib.ESTIMATE)
        h.set(_lib.NOISY, 0, np.ones(x.shape))
        h.ft_error(x)
        h.simulate(1e6, 3)
        got = np.concatenate([h.get(_lib.NOISELESS, k) for k in range(2)])
        assert rel_l2(got, want) < 1e-12
    h.close()
