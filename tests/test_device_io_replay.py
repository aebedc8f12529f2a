"""The device-buffer entry points (lsted_deconv_*_dev) on the CPU replay of the
kernel bodies: every one gives the bits of its host twin -- both precisions,
float32 and float64 caller buffers, 16-byte-aligned and element-aligned-only
buffers, untiled and tiled handles, a ragged size.  In the replay a "device"
pointer is host memory, so numpy arrays stand in for CUDA tensors.  Also the
argument checks the library makes before anything runs, and the rejections the
Python layer makes before any call crosses into the library."""
import ctypes

import numpy as np
import pytest

import emul_support
from rescan_line_sted_b200 import _lib

SHAPE = (77, 91)        # 7007 pixels: the last 16-byte group of either dtype is partial
K = 3


@pytest.fixture(scope='module')
def lib():
    return emul_support.emulator_library()


def buffer(n, dtype, offset):
    """n elements at `offset` elements past a 64-byte boundary (1: element-aligned only)."""
    item = np.dtype(dtype).itemsize
    raw = np.zeros(n * item + 64 + offset * item + 64, dtype=np.uint8)
    start = (-raw.ctypes.data) % 64 + offset * item
    out = raw[start:start + n * item].view(dtype)
    assert (out.ctypes.data % 16 == 0) == (offset == 0)
    return out


def filled(values, dtype, offset):
    b = buffer(values.size, dtype, offset)
    b[...] = values.ravel()
    return b


def bits(dtype):
    return 32 if dtype == np.float32 else 64


def make_handle(lib, precision, tiled):
    rng = np.random.default_rng(11)
    psfs = rng.random((K, 9, 11))
    return _lib.DeconvHandle(lib, psfs, SHAPE, precision=precision,
                             tile_fft_len=64 if tiled else 0)


def host_result(a, dtype):
    """What a caller of the host entry point holds after converting to `dtype`."""
    return np.asarray(a, dtype=np.float64).astype(dtype).ravel()


CASES = [pytest.param(p, t, id='fp%d-%s' % (p, 'tiled' if t else 'untiled'))
         for p in (32, 64) for t in (False, True)]
BUFFERS = [pytest.param(d, o, id='%s-off%d' % (np.dtype(d).name, o))
           for d in (np.float32, np.float64) for o in (0, 1)]


@pytest.mark.parametrize('dtype,offset', BUFFERS)
@pytest.mark.parametrize('precision,tiled', CASES)
def test_dev_entry_points_equal_host_twins(lib, precision, tiled, dtype, offset):
    h = make_handle(lib, precision, tiled)
    if tiled:
        assert (h.info().tiles_y, h.info().tiles_x) == (2, 2)
    npix = SHAPE[0] * SHAPE[1]
    rng = np.random.default_rng(5)
    # inputs hold values of the caller dtype; the host twin is fed the same values in float64
    x = rng.random((1,) + SHAPE).astype(dtype).astype(np.float64)
    y = rng.random((K,) + SHAPE).astype(dtype).astype(np.float64)
    nbits = bits(dtype)

    # H
    xd, out = filled(x, dtype, offset), buffer(K * npix, dtype, offset)
    lib.call('lsted_deconv_H_dev', h._h, xd.ctypes.data, out.ctypes.data, nbits, None)
    np.testing.assert_array_equal(out, host_result(h.H(x), dtype))
    # H_t, normalised and not
    yd = filled(y, dtype, offset)
    for normalize in (0, 1):
        out = buffer(npix, dtype, offset)
        lib.call('lsted_deconv_Ht_dev', h._h, yd.ctypes.data, out.ctypes.data, nbits,
                 normalize, None)
        np.testing.assert_array_equal(out, host_result(h.Ht(y, bool(normalize)), dtype))

    # upload_object_dev + simulate == create_data (same seed: the same Philox field)
    obj = (rng.random((1,) + SHAPE) + 0.1).astype(dtype).astype(np.float64)
    h.create_data(obj, 1e6, 17)
    want = {w: [h.get(w, k).copy() for k in range(K if w in (1, 2) else 1)] for w in (0, 1, 2)}
    h.set(_lib.NOISY, 0, np.zeros((1,) + SHAPE))
    od = filled(obj, dtype, offset)
    lib.call('lsted_deconv_upload_object_dev', h._h, od.ctypes.data, nbits, None)
    h.simulate(1e6, 17)
    for w, arrays in want.items():
        for k, a in enumerate(arrays):
            np.testing.assert_array_equal(h.get(w, k), a)

    # get_dev of all five arrays (per PSF k for the measurements)
    h.iterate(2)
    for which in range(5):
        for k in range(K if which in (_lib.NOISELESS, _lib.NOISY) else 1):
            out = buffer(npix, dtype, offset)
            lib.call('lsted_deconv_get_dev', h._h, which, k, out.ctypes.data, nbits, None)
            np.testing.assert_array_equal(out, host_result(h.get(which, k), dtype))

    # set_dev equals set of the same values (read back through the host path)
    for which in range(5):
        for k in range(K if which in (_lib.NOISELESS, _lib.NOISY) else 1):
            v = (rng.random((1,) + SHAPE) + 0.5).astype(dtype).astype(np.float64)
            h.set(which, k, v)
            want = h.get(which, k).copy()
            h.set(which, k, np.zeros((1,) + SHAPE))
            vd = filled(v, dtype, offset)
            lib.call('lsted_deconv_set_dev', h._h, which, k, vd.ctypes.data, nbits, None)
            np.testing.assert_array_equal(h.get(which, k), want)
    # the estimate set through the device path iterates like the host one
    est = (rng.random((1,) + SHAPE) + 0.5).astype(dtype).astype(np.float64)
    h.set(_lib.ESTIMATE, 0, est)
    h.iterate(1)
    want = h.get(_lib.ESTIMATE).copy()
    ed = filled(est, dtype, offset)
    lib.call('lsted_deconv_set_dev', h._h, _lib.ESTIMATE, 0, ed.ctypes.data, nbits, None)
    h.iterate(1)
    np.testing.assert_array_equal(h.get(_lib.ESTIMATE), want)
    h.close()


def status(lib, name, *args):
    return getattr(lib.cdll, name)(*args)


def test_dev_argument_checks(lib):
    h = make_handle(lib, 32, False)
    npix = SHAPE[0] * SHAPE[1]
    x, out = buffer(npix, np.float32, 0), buffer(K * npix, np.float32, 0)
    for bad in (0, 16, 33, 128):
        assert status(lib, 'lsted_deconv_H_dev', h._h, x.ctypes.data, out.ctypes.data, bad, None) == 1
        assert 'dtype' in lib.last_error()
        assert status(lib, 'lsted_deconv_get_dev', h._h, 0, 0, out.ctypes.data, bad, None) == 1
    # a pointer that is not aligned to its element type
    raw = np.zeros(8 * npix + 16, dtype=np.uint8)
    assert status(lib, 'lsted_deconv_upload_object_dev', h._h, raw.ctypes.data + 1, 64, None) == 1
    assert 'aligned' in lib.last_error()
    assert status(lib, 'lsted_deconv_Ht_dev', h._h, raw.ctypes.data + 2, out.ctypes.data, 32, 1,
                  None) == 1
    assert status(lib, 'lsted_deconv_set_dev', h._h, 0, 0, None, 32, None) == 1
    assert 'null' in lib.last_error()
    # array selectors follow the host twins
    assert status(lib, 'lsted_deconv_get_dev', h._h, 5, 0, out.ctypes.data, 32, None) == 1
    assert status(lib, 'lsted_deconv_get_dev', h._h, _lib.NOISY, K, out.ctypes.data, 32, None) == 1
    assert status(lib, 'lsted_deconv_set_dev', h._h, _lib.ESTIMATE, 1, x.ctypes.data, 32, None) == 1
    h.close()


# ---- Python-level rejections: no GPU needed, nothing reaches the library (a Deconvolver
# takes any (1, Ny, Nx) as its first image, so 'wrong-size' applies to a handle only) ----
try:
    import torch
except ImportError:          # the numpy product works without torch; these tests need it
    torch = None
needs_torch = pytest.mark.skipif(torch is None, reason='torch is not importable')


class _NoLibrary:
    """Stands in for the library: any call through it is a test failure."""
    def __getattr__(self, name):
        raise AssertionError('the library was called: %s' % name)


def tensor_handle():
    h = _lib.DeconvHandle.__new__(_lib.DeconvHandle)
    h.lib, h._h = _NoLibrary(), ctypes.c_void_p()
    h.K, h.ny, h.nx, h.Ny, h.Nx, h.precision, h.device = K, 9, 11, SHAPE[0], SHAPE[1], 32, 0
    return h


BAD_TENSORS = [
    pytest.param(lambda: torch.ones((1,) + SHAPE), ValueError, 'CUDA', id='cpu'),
    pytest.param(lambda: torch.ones(SHAPE), ValueError, 'shape', id='2d'),
    pytest.param(lambda: torch.ones((1, 76, 91)), ValueError, 'shape', id='wrong-size'),
    pytest.param(lambda: torch.ones((1,) + SHAPE, dtype=torch.int32), TypeError, 'float', id='int32'),
    pytest.param(lambda: torch.ones((1,) + SHAPE, dtype=torch.float16), TypeError, 'float', id='half'),
    pytest.param(lambda: torch.ones((1, SHAPE[1], SHAPE[0])).transpose(1, 2), ValueError,
                 'contiguous', id='non-contiguous'),
    pytest.param(lambda: np.ones((1,) + SHAPE), TypeError, 'Tensor', id='numpy'),
]


@needs_torch
@pytest.mark.parametrize('make,exc,words', BAD_TENSORS)
def test_handle_rejects_bad_tensors(make, exc, words):
    h = tensor_handle()
    for call in (lambda t: h.H_tensor(t), lambda t: h.set_tensor(_lib.ESTIMATE, 0, t),
                 lambda t: h.upload_object_tensor(t), lambda t: h.get_tensor(0, 0, out=t)):
        with pytest.raises(exc, match=words):
            call(make())


@needs_torch
def test_handle_rejects_ht_input_of_wrong_count():
    h = tensor_handle()
    with pytest.raises(ValueError, match='shape'):
        h.Ht_tensor(torch.ones((K - 1,) + SHAPE))


@needs_torch
@pytest.mark.parametrize('make,exc,words', [p for p in BAD_TENSORS if p.id not in ('numpy', 'wrong-size')])
def test_deconvolver_rejects_bad_tensors(tmp_path, make, exc, words):
    from rescan_line_sted_b200 import line_sted_tools as st
    d = st.Deconvolver([np.ones((1, 3, 3))] * K, output_prefix=str(tmp_path) + '/x_',
                       verbose=False)
    for call in (lambda t: d.H(t), lambda t: d.H_t([t] * K),
                 lambda t: d.create_data_from_object(t),
                 lambda t: setattr(d, 'estimate', t),
                 lambda t: setattr(d, 'noisy_measurement', [t] * K)):
        with pytest.raises(exc, match=words):
            call(make())
    assert d._handle is None          # rejected before any handle was built


@needs_torch
def test_deconvolver_tensor_accessor_names(tmp_path):
    from rescan_line_sted_b200 import line_sted_tools as st
    d = st.Deconvolver([np.ones((1, 3, 3))], output_prefix=str(tmp_path) + '/x_', verbose=False)
    with pytest.raises(ValueError, match='estimate'):
        d.tensor('psfs')
    with pytest.raises(AttributeError, match="no attribute 'estimate'"):
        d.tensor('estimate')
    with pytest.raises(TypeError, match='dtype'):
        d.tensor('estimate', dtype=torch.int64)
