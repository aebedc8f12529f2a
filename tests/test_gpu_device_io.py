"""CUDA tensors in and out of a Deconvolver handle (the lsted_deconv_*_dev entry
points): the same bits as the host path, ordered on the caller's stream without
blocking the host, and every bad buffer refused before anything is launched."""
import ctypes
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from rescan_line_sted_b200 import _lib

pytestmark = pytest.mark.gpu
torch = pytest.importorskip('torch')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PER_PSF = (_lib.NOISELESS, _lib.NOISY)


def sym_psfs(K, ny, nx, seed=0):
    """Point-symmetric PSFs of odd size (what the reference builds): centred real OTFs."""
    p = np.random.default_rng(seed).random((K, ny, nx))
    return p + p[:, ::-1, ::-1]


# (image shape, PSFs, tile FFT length)
CASES = [
    pytest.param((2048, 2048), (4, 107, 107), 0, id='2048-plan2160'),
    pytest.param((128, 128), (3, 9, 9), 0, id='128-generic'),
    pytest.param((77, 91), (3, 9, 11), 0, id='77x91'),
    pytest.param((150, 170), (3, 9, 11), 64, id='tiled'),
]
DTYPES = [pytest.param(torch.float32, id='f32'), pytest.param(torch.float64, id='f64')]


def dev(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a)).to(device='cuda:0', dtype=dtype)


def host_as(a, dtype):
    """A host-path result as the caller converts it to `dtype` (one rounding)."""
    return torch.as_tensor(np.array(a, dtype=np.float64)).to(dtype)


def same(t, host, dtype=None):
    t = t.cpu()
    return torch.equal(t, host_as(host, dtype or t.dtype).reshape(t.shape))


@pytest.fixture(scope='module')
def lib():
    return _lib.get()


@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('precision', [32, 64])
@pytest.mark.parametrize('shape,psf_shape,tile', CASES)
def test_bits_equal_host_path(lib, shape, psf_shape, tile, precision, dtype):
    K = psf_shape[0]
    h = _lib.DeconvHandle(lib, sym_psfs(*psf_shape), shape, precision=precision, tile_fft_len=tile)
    g = torch.Generator(device='cuda:0').manual_seed(1)
    x = torch.rand((1,) + shape, generator=g, device='cuda:0', dtype=dtype)
    y = torch.rand((K,) + shape, generator=g, device='cuda:0', dtype=dtype)
    xh, yh = x.double().cpu().numpy(), y.double().cpu().numpy()
    assert same(h.H_tensor(x), h.H(xh))
    assert same(h.Ht_tensor(y, normalize=False), h.Ht(yh, False))
    assert same(h.Ht_tensor(y, normalize=True), h.Ht(yh, True))

    obj = torch.rand((1,) + shape, generator=g, device='cuda:0', dtype=dtype) + 0.1
    h.create_data(obj.double().cpu().numpy(), 1e9, 3)
    h.iterate(3)
    for which in range(5):
        for k in range(K if which in PER_PSF else 1):
            assert same(h.get_tensor(which, k, dtype), h.get(which, k)), (which, k)
    for which in range(5):
        for k in range(K if which in PER_PSF else 1):
            v = torch.rand((1,) + shape, generator=g, device='cuda:0', dtype=dtype) + 0.5
            h.set(which, k, v.double().cpu().numpy())
            want = h.get(which, k).copy()
            h.set(which, k, np.zeros((1,) + shape))
            h.set_tensor(which, k, v)
            assert np.array_equal(h.get(which, k), want), (which, k)
    h.close()


@pytest.mark.parametrize('shape,psf_shape,precision', [
    pytest.param((2048, 2048), (16, 107, 107), 'fp32', id='2048-K16-fp32'),
    pytest.param((128, 128), (4, 107, 107), 'fp64', id='128-fp64'),
])
@pytest.mark.parametrize('dtype', DTYPES)
def test_whole_frame_equals_numpy_path(monkeypatch, tmp_path, shape, psf_shape, precision, dtype):
    monkeypatch.setenv('LSTED_PRECISION', precision)
    from rescan_line_sted_b200 import line_sted_tools as st
    psfs = [p[None] for p in sym_psfs(*psf_shape, seed=2)]
    obj = torch.rand((1,) + shape, generator=torch.Generator(device='cuda:0').manual_seed(4),
                     device='cuda:0', dtype=dtype) + 0.05
    a = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/a_', verbose=False)
    b = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/b_', verbose=False)
    a.create_data_from_object(obj, total_brightness=1e10, random_seed=77)
    b.create_data_from_object(obj.double().cpu().numpy(), total_brightness=1e10, random_seed=77)
    a.iterate_many(8)
    b.iterate_many(8)
    est = a.tensor('estimate')
    assert est.dtype == torch.float64 and est.shape == (1,) + shape
    assert same(est, b.estimate)
    noisy = a.tensor('noisy_measurement')
    assert len(noisy) == psf_shape[0]
    for t, want in zip(noisy, b.noisy_measurement):
        assert t.shape == (1,) + shape and same(t, want)   # the Philox field
    assert same(a.tensor('true_object', torch.float32), b.true_object)
    assert same(a.tensor('H_t_normalization'), b.H_t_normalization)


def test_stream_order_without_host_sync(tmp_path):
    from rescan_line_sted_b200 import line_sted_tools as st
    shape = (1, 128, 128)
    d = st.Deconvolver([p[None] for p in sym_psfs(3, 9, 9)], output_prefix=str(tmp_path) + '/s_',
                       verbose=False)
    src = torch.rand(shape, device='cuda:0')
    d.H(src)                                       # builds the handle and its temporaries
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        x = torch.empty_like(src)
        torch.cuda._sleep(int(2e9))
        x.copy_(src)                               # the kernel that fills the input
        out = d.H(x)
        pending = not s.query()
    s.synchronize()
    assert pending, 'H of a tensor waited for the stream'
    want = d.H(src.double().cpu().numpy())
    assert all(same(o, w) for o, w in zip(out, want))


def test_inputs_may_be_reused_at_once(tmp_path):
    from rescan_line_sted_b200 import line_sted_tools as st
    shape = (1, 128, 128)
    d = st.Deconvolver([p[None] for p in sym_psfs(3, 9, 9)], output_prefix=str(tmp_path) + '/r_',
                       verbose=False)
    src = torch.rand((3,) + shape[1:], device='cuda:0')
    want = d.H_t([src[k:k + 1].double().cpu().numpy() for k in range(3)])
    want_raw = d._handle.Ht(src.double().cpu().numpy(), False)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(1e9))
        out = d.H_t([src[k:k + 1].clone() for k in range(3)])    # the list dies here
        junk = [torch.full(shape, float('nan'), device='cuda:0') for _ in range(4)]
        y = src.clone()
        out_raw = d._handle.Ht_tensor(y, normalize=False)
        del y
        junk.append(torch.full((3,) + shape[1:], float('nan'), device='cuda:0'))
    s.synchronize()
    assert same(out, want) and same(out_raw, want_raw)
    del junk


def test_views_at_an_element_offset(lib):
    shape = (77, 91)
    npix = shape[0] * shape[1]
    h = _lib.DeconvHandle(lib, sym_psfs(3, 9, 11), shape, precision=32)
    for dtype in (torch.float32, torch.float64):
        base = torch.rand(npix + 1, device='cuda:0', dtype=dtype)
        x = base[1:].view((1,) + shape)
        assert x.storage_offset() == 1 and x.data_ptr() % 16 != 0
        assert same(h.H_tensor(x), h.H(x.double().cpu().numpy()))
        h.set_tensor(_lib.ESTIMATE, 0, x)
        buf = torch.zeros(npix + 1, device='cuda:0', dtype=dtype)
        h.get_tensor(_lib.ESTIMATE, out=buf[1:].view((1,) + shape))
        assert buf[0].item() == 0 and same(buf[1:], h.get(_lib.ESTIMATE))


def test_host_and_misplaced_pointers_are_refused(lib):
    shape = (64, 64)
    npix = shape[0] * shape[1]
    h = _lib.DeconvHandle(lib, sym_psfs(3, 9, 9), shape, precision=32)
    out = torch.empty((3,) + shape, device='cuda:0', dtype=torch.float64)
    x = torch.rand((1,) + shape, device='cuda:0', dtype=torch.float64)
    host = np.zeros(npix)
    pinned = _lib.pinned_empty((1,) + shape)
    for p in (host.ctypes.data, pinned.ctypes.data):
        assert lib.cdll.lsted_deconv_H_dev(h._h, ctypes.c_void_p(p), ctypes.c_void_p(out.data_ptr()),
                                           64, None) == 1
        assert 'host memory' in lib.last_error()
        assert lib.cdll.lsted_deconv_H_dev(h._h, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(p),
                                           64, None) == 1
    _lib.pinned_free(pinned)
    # a stream being captured into a CUDA graph
    g, s = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(g, stream=s, capture_error_mode='relaxed'):
        code = lib.cdll.lsted_deconv_H_dev(h._h, ctypes.c_void_p(x.data_ptr()),
                                           ctypes.c_void_p(out.data_ptr()), 64,
                                           ctypes.c_void_p(s.cuda_stream))
    assert code == 4 and 'captured' in lib.last_error()
    if torch.cuda.device_count() > 1:
        other = torch.rand((1,) + shape, device='cuda:1', dtype=torch.float64)
        with pytest.raises(ValueError, match='cuda:1'):
            h.H_tensor(other)
        assert lib.cdll.lsted_deconv_H_dev(h._h, ctypes.c_void_p(other.data_ptr()),
                                           ctypes.c_void_p(out.data_ptr()), 64, None) == 1
        assert 'device 1' in lib.last_error()
    # the handle still works
    assert same(h.H_tensor(x), h.H(x.cpu().numpy()))


OVERRUN = textwrap.dedent('''
    import ctypes, sys
    import numpy as np, torch
    sys.path.insert(0, sys.argv[1])
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    shape = (512, 512)
    npix = shape[0] * shape[1]
    h = _lib.DeconvHandle(lib, np.ones((3, 9, 9)), shape, precision=32)
    x = torch.rand((1,) + shape, device='cuda:0')
    short = torch.empty(3 * npix - (1 << 18), device='cuda:0')      # 1 MiB short of K images
    ok_out = torch.empty((3,) + shape, device='cuda:0')
    bad = lib.cdll.lsted_deconv_H_dev(h._h, ctypes.c_void_p(x.data_ptr()),
                                      ctypes.c_void_p(short.data_ptr()), 32, None)
    msg = lib.last_error()
    good = lib.cdll.lsted_deconv_H_dev(h._h, ctypes.c_void_p(x.data_ptr()),
                                       ctypes.c_void_p(ok_out.data_ptr()), 32, None)
    torch.cuda.synchronize()
    print('STATUS', bad, good, msg)
''')


def test_range_past_the_allocation_is_refused():
    env = dict(os.environ, PYTORCH_NO_CUDA_MEMORY_CACHING='1')
    r = subprocess.run([sys.executable, '-c', OVERRUN, ROOT], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith('STATUS')][0]
    bad, good, msg = line.split(' ', 3)[1:]
    assert (bad, good) == ('1', '0'), line
    assert 'allocation' in msg


def test_handle_unaffected_by_device_calls(tmp_path):
    from rescan_line_sted_b200 import line_sted_tools as st
    shape = (1, 96, 112)
    psfs = [p[None] for p in sym_psfs(3, 9, 9, seed=5)]
    rng = np.random.default_rng(8)
    obj = rng.random(shape) + 0.1
    x = rng.random(shape)
    a = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/a_', verbose=False)
    b = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/b_', verbose=False)
    for d in (a, b):
        d.create_data_from_object(obj, total_brightness=1e9, random_seed=9)
        d.iterate()
    xt = dev(x, torch.float32)
    a.H(xt)
    a.H_t([xt] * 3, normalize=False)
    a.tensor('estimate')
    a.tensor('noiseless_measurement')
    for d in (a, b):
        d.H(x)
        d.iterate()
        d.iterate_many(3)
    assert a.num_iterations == b.num_iterations == 5
    assert isinstance(a.estimate, np.ndarray)
    assert np.array_equal(a.estimate, b.estimate)
    assert np.array_equal(a.H_t_normalization, b.H_t_normalization)
    for u, v in zip(a.noisy_measurement, b.noisy_measurement):
        assert np.array_equal(u, v)
