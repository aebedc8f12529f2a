"""The local error metrics of _local_error on a CPU stand-in for the engine: float32 scipy.fft
convolutions against float64 ones.  An honest fp32 transform passes every bound; each fault a
single CTA or tile could make passes the old whole-stack check (rel-L2 < 1e-5) and fails the local
one, with a message that names the orientation and the unit."""
import numpy as np
import pytest
import scipy.fft

from _local_error import Geometry, LocalErrors

OLD_TOL = 1e-5
N, L = 2048, 2160                       # the headline frame and its transform length
GEOM = Geometry(L, L, 4, 2, 1, 1, 0, 0)


def conv(x, p, n, dtype):
    """Linear convolution of each x[k] with p[k] over n x n transforms in `dtype`, cropped like
    fftconvolve_same."""
    s = (p.shape[-2] - 1) // 2, (p.shape[-1] - 1) // 2
    X = scipy.fft.rfft2(x.astype(dtype), s=(n, n))
    P = scipy.fft.rfft2(p.astype(dtype), s=(n, n))
    y = scipy.fft.irfft2(X * P, s=(n, n))
    return y[..., s[0]:s[0] + x.shape[-2], s[1]:s[1] + x.shape[-1]].astype(np.float64)


def stand_in(shape, K, n, psf=21, seed=0):
    rng = np.random.default_rng(seed)
    x = rng.random((1,) + shape) + 0.1
    p = rng.random((K, psf, psf))
    return conv(x, p, n, np.float32), conv(x, p, n, np.float64)


@pytest.fixture(scope='module')
def headline():
    """2048^2, one random 21 x 21 PSF, transforms of length 2160: (fp32 result, fp64 result)."""
    return stand_in((N, N), 1, L)


def rel_l2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def failures(got, want, geom, precision=32):
    return LocalErrors(got, want, geom, precision).failures('fault')


def test_fp32_fft_passes_every_bound(headline):
    got, want = headline
    r = LocalErrors(got, want, GEOM, 32)
    print(r.report('fp32 scipy.fft at 2048^2'))
    assert not r.failures('fp32 scipy.fft')


@pytest.mark.parametrize('shape,K,n,geom', [
    ((300, 500), 4, 540, Geometry(540, 540, 4, 1, 1, 1, 0, 0)),
    ((150, 170), 3, 192, Geometry(64, 64, 4, 2, 3, 4, 56, 54)),
])
def test_fp32_fft_passes_every_bound_on_other_geometries(shape, K, n, geom):
    got, want = stand_in(shape, K, n, psf=9)
    r = LocalErrors(got, want, geom, 32)
    print(r.report('fp32 scipy.fft %s' % (shape,)))
    assert not r.failures('fp32 scipy.fft')


def spectral_fault(want, bin0, nbins, scale, Lx=L):
    """Scale bins bin0 .. bin0 + nbins - 1 of the row spectrum (zero-padded to Lx)."""
    f = np.fft.rfft(want, n=Lx, axis=-1)
    f[..., bin0:bin0 + nbins] *= scale
    return np.fft.irfft(f, n=Lx, axis=-1)[..., :want.shape[-1]]


def faulty(want, kind):
    got = want.copy()
    if kind == 'row pair':
        got[0, 1000:1002] *= 1 + 2.5e-4
    elif kind == 'pixel':
        got[0, 700, 1300] *= 1.01
    elif kind == 'column block 600':
        got = spectral_fault(want, 600, 4, 1 + 1e-3)
    elif kind == 'column block 1000':
        got = spectral_fault(want, 1000, 4, 1 + 1e-2)
    elif kind == 'stale patch':             # a 32 x 32 patch of the result of another input
        rng = np.random.default_rng(1)
        other = want * (1 + 4e-4 * rng.standard_normal(want.shape))
        got[0, 900:932, 500:532] = other[0, 900:932, 500:532]
    return got


# (fault, the unit the message must name)
FAULTS = {
    'row pair': 'k = 0, rows 1000-1003',
    'pixel': 'k = 0, pixel (700, 1300)',
    'column block 600': 'k = 0, column block 150 (bins 600-603)',
    'column block 1000': 'k = 0, column block 250 (bins 1000-1003)',
    'stale patch': 'k = 0, pixel (9',
}


@pytest.mark.parametrize('kind', sorted(FAULTS))
def test_fault_passes_old_check_and_fails_the_local_one(headline, kind):
    _, want = headline
    got = faulty(want, kind)
    assert rel_l2(got, want) < OLD_TOL
    msgs = failures(got, want, GEOM)
    assert msgs, kind
    print('\n'.join(msgs))
    assert any(FAULTS[kind] in m for m in msgs), (kind, msgs)


def test_one_orientation_of_sixteen():
    """One of K = 16 orientations scaled by 1 + 2e-5: a quarter of that in the whole-stack
    rel-L2."""
    got, want = stand_in((256, 256), 16, 288)
    got = want.copy()
    got[11] *= 1 + 2e-5
    assert rel_l2(got, want) < OLD_TOL
    msgs = failures(got, want, Geometry(288, 288, 4, 2, 1, 1, 0, 0))
    assert any(m.startswith('fault: orientation k = 11:') for m in msgs), msgs


def test_one_tile_of_a_tiled_layout():
    """A 3 x 4 grid of 64-point windows (56 x 54 output pixels each); tile 6 scaled by
    1 + 2e-5."""
    geom = Geometry(64, 64, 4, 2, 3, 4, 56, 54)
    _, want = stand_in((150, 170), 1, 192, psf=9)
    got = want.copy()
    got[0, 56:112, 108:162] *= 1 + 2e-5
    assert rel_l2(got, want) < OLD_TOL
    msgs = failures(got, want, geom)
    assert any('tile k = 0, tile 6 (rows 56-111, columns 108-161)' in m for m in msgs), msgs


def test_estimate_metric_needs_its_floor_on_dark_objects():
    """Per-pixel estimate error against |want| + f * max|want|: an fp32 Richardson-Lucy step on
    beads on a dark background passes, one pixel 1 % off fails and is named."""
    rng = np.random.default_rng(3)
    x = np.zeros((1, 300, 320))
    x[0, rng.integers(0, 300, 40), rng.integers(0, 320, 40)] = 1.0
    p = rng.random((2, 9, 9))
    geom = Geometry(320, 360, 4, 2, 1, 1, 0, 0)

    def rl_step(dtype):
        y = conv(x, p, 360, np.float64) + 1e-3          # noiseless measurements
        est = np.ones_like(x)
        ratio = y / np.maximum(conv(est, p, 360, dtype), 1e-12)
        return est * conv(ratio, p, 360, dtype).sum(0, keepdims=True) / conv(
            np.ones_like(y), p, 360, dtype).sum(0, keepdims=True)
    got, want = rl_step(np.float32), rl_step(np.float64)
    r = LocalErrors(got, want, geom, 32, estimate=True)
    print(r.report('fp32 RL step, dark object'))
    assert not r.failures('fp32 RL step')
    bad = want.copy()
    bad[0, 150, 160] *= 1.01
    msgs = LocalErrors(bad, want, geom, 32, estimate=True).failures('fault')
    assert any('k = 0, pixel (150, 160)' in m for m in msgs), msgs
