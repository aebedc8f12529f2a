"""Parity of the CUDA Deconvolver (through the C ABI / ctypes mirror) with
the CPU oracle and the golden fixtures of the unmodified reference.
Tolerances (BASELINE.json north_star): rel-L2 <= 1e-5 in fp32, <= 1e-12 in
fp64 for noise-free images; iterated estimates get one decade more."""
import json
import os

import numpy as np
import pytest

from _local_error import check_local, local_errors
from oracle import line_sted_oracle as orc

pytestmark = pytest.mark.gpu

TOL = {'fp32': 1e-5, 'fp64': 1e-12}


def rel_l2(a, b):
    den = np.linalg.norm(np.ravel(b))
    return np.linalg.norm(np.ravel(a) - np.ravel(b)) / (den if den > 0 else 1.0)


@pytest.fixture(scope='module')
def st():
    from rescan_line_sted_b200 import line_sted_tools
    return line_sted_tools


@pytest.fixture(scope='module')
def fig2(golden_dir):
    return np.load(os.path.join(golden_dir, 'fig2_2p0x_lr.npz'))


@pytest.fixture(params=['fp64', 'fp32'])
def precision(request, monkeypatch):
    monkeypatch.setenv('LSTED_PRECISION', request.param)
    return request.param


def test_golden_forward_and_rl(st, fig2, precision, tmp_path):
    tol = TOL[precision]
    psfs = [p[None] for p in fig2['psfs']]
    d = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/g_', verbose=False)
    d.create_data_from_object(fig2['object_u8'].astype(np.float64),
                              total_brightness=5e10, random_seed=0)
    assert rel_l2(np.concatenate(d.noiseless_measurement), fig2['noiseless']) < tol
    d.noisy_measurement = [m[None] for m in fig2['noisy']]  # injected field
    d.iterate()
    assert rel_l2(d.H_t_normalization, fig2['H_t_normalization']) < tol
    assert rel_l2(d.estimate, fig2['estimate_1']) < tol
    for _ in range(7):
        d.iterate()
    assert rel_l2(d.estimate, fig2['estimate_8']) < 10 * tol
    assert d.num_iterations == 8


@pytest.mark.parametrize('shape,pshape', [((1, 33, 40), (1, 9, 9)),
                                          ((1, 128, 128), (1, 107, 107)),
                                          ((1, 160, 160), (1, 107, 107)),
                                          ((1, 7, 300), (1, 11, 5)),
                                          ((1, 50, 31), (1, 8, 6)),
                                          ((1, 1, 64), (1, 1, 9)),
                                          ((1, 5, 9), (1, 11, 11))])
def test_H_and_Ht_ragged_shapes(st, precision, shape, pshape, tmp_path):
    tol = TOL[precision]
    rng = np.random.default_rng(3)
    psfs = [rng.random(pshape) for _ in range(3)]
    d = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/h_', verbose=False)
    o = orc.Deconvolver(psfs)
    x = rng.random(shape)
    got, want = d.H(x), o.H(x)
    for a, b in zip(got, want):
        assert a.shape == b.shape
        assert rel_l2(a, b) < tol
    y = [rng.random(shape) for _ in psfs]
    Ht, Ht_want = d.H_t(y, normalize=False), o.H_t(y, normalize=False)
    assert rel_l2(Ht, Ht_want) < tol
    info, bits = d._handle.info(), int(precision[2:])
    label = 'ragged %s psf %s' % (shape[1:], pshape[1:])
    check_local([(label + ' H', local_errors(np.concatenate(got), np.concatenate(want), info, bits)),
                 (label + ' Ht', local_errors(Ht, Ht_want, info, bits))])
    assert rel_l2(d.H_t(y), o.H_t(y)) < tol
    assert rel_l2(d.H_t_normalization, o.H_t_normalization) < tol


def test_mixed_psf_sizes(st, precision, tmp_path):
    rng = np.random.default_rng(4)
    psfs = [rng.random((1, 9, 9)), rng.random((1, 7, 11)), rng.random((1, 4, 6))]
    d = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/m_', verbose=False)
    o = orc.Deconvolver(psfs)
    x = rng.random((1, 40, 33))
    for a, b in zip(d.H(x), o.H(x)):
        assert rel_l2(a, b) < TOL[precision]


def test_rl_random_object_vs_oracle(st, precision, tmp_path):
    tol = TOL[precision]
    rng = np.random.default_rng(11)
    psfs = [rng.random((1, 9, 9)), rng.random((1, 9, 9)), rng.random((1, 7, 11))]
    obj = rng.random((1, 33, 40)) + 0.1
    d = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/r_', verbose=False)
    o = orc.Deconvolver(psfs)
    d.create_data_from_object(obj, total_brightness=1e6, random_seed=3)
    o.create_data_from_object(obj, total_brightness=1e6, random_seed=3)
    assert rel_l2(d.true_object, o.true_object) < tol
    d.noisy_measurement = o.noisy_measurement
    for _ in range(5):
        d.iterate(), o.iterate()
    assert rel_l2(d.estimate, o.estimate) < 10 * tol


def test_exact_clip_mode_matches_too(st, fig2, monkeypatch, tmp_path):
    monkeypatch.setenv('LSTED_PRECISION', 'fp64')
    monkeypatch.setenv('LSTED_EXACT_CLIP', '1')
    psfs = [p[None] for p in fig2['psfs']]
    d = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/e_', verbose=False)
    d.create_data_from_object(fig2['object_u8'].astype(np.float64),
                              total_brightness=5e10, random_seed=0)
    d.noisy_measurement = [m[None] for m in fig2['noisy']]
    for _ in range(8):
        d.iterate()
    assert rel_l2(d.estimate, fig2['estimate_8']) < 1e-11


def test_poisson_statistics_in_kernel(st, monkeypatch, tmp_path):
    """In-kernel Philox Poisson: mean and variance match the noiseless
    image (statistical parity; the reference uses MT19937)."""
    monkeypatch.setenv('LSTED_PRECISION', 'fp64')
    rng = np.random.default_rng(5)
    psfs = [np.ones((1, 5, 5)) / 25.]
    obj = np.ones((1, 256, 256)) + 0.0 * rng.random((1, 256, 256))
    d = st.Deconvolver(psfs, output_prefix=str(tmp_path) + '/p_', verbose=False)
    for lam in (0.5, 4.0, 9.5, 30.0, 1e3, 2e7):
        d.create_data_from_object(obj, total_brightness=lam * obj.size,
                                  random_seed=7)
        nl = d.noiseless_measurement[0][0, 8:-8, 8:-8]
        ny = d.noisy_measurement[0][0, 8:-8, 8:-8]
        assert np.all(ny > 0)                       # '+ 1e-9': no zeros (ref:510)
        ny = ny - 1e-9
        assert np.allclose(nl, lam, rtol=1e-9)
        n = nl.size
        assert np.abs(ny - np.round(ny)).max() < 1e-6 * max(1.0, lam)
        ny = np.round(ny)
        assert ny.min() >= 0
        assert abs(ny.mean() - lam) < 5 * np.sqrt(lam / n)
        assert abs(ny.var() / lam - 1) < 5 * np.sqrt(2.0 / n) + 1e-3
    # different seeds give different fields, same seed repeats exactly
    d.create_data_from_object(obj, total_brightness=100. * obj.size, random_seed=1)
    a = d.noisy_measurement[0]
    d.create_data_from_object(obj, total_brightness=100. * obj.size, random_seed=1)
    assert np.array_equal(a, d.noisy_measurement[0])
    d.create_data_from_object(obj, total_brightness=100. * obj.size, random_seed=2)
    assert not np.array_equal(a, d.noisy_measurement[0])


def test_attribute_protocol(st, tmp_path):
    rng = np.random.default_rng(1)
    d = st.Deconvolver([rng.random((1, 5, 5))], output_prefix=str(tmp_path) + '/a_',
                       verbose=False)
    assert not hasattr(d, 'estimate') and not hasattr(d, 'noisy_measurement')
    assert not hasattr(d, 'H_t_normalization')
    with pytest.raises(AssertionError):
        d.create_data_from_object(np.ones((16, 16)))             # not 3-D
    with pytest.raises(AssertionError):
        d.create_data_from_object(np.ones((1, 16, 16), dtype=np.float32))
    d.create_data_from_object(np.ones((1, 16, 16)), total_brightness=1e4)
    assert hasattr(d, 'noisy_measurement') and not hasattr(d, 'estimate')
    d.iterate()
    assert d.estimate.shape == (1, 16, 16) and d.estimate.dtype == np.float64
    assert hasattr(d, 'H_t_normalization')
    d.record_data()
    d.record_iteration()
    assert os.path.exists(str(tmp_path) + '/a_estimate_history.tif')
    assert os.path.exists(str(tmp_path) + '/a_noisy_measurement.tif')


def test_large_results_come_back_in_recycled_pinned_buffers():
    """Arrays of >= 1 MB read back from the handle live in page-locked memory from a pool:
    they behave like any numpy array, stay valid while referenced, and their buffer is
    reused once they are garbage-collected."""
    import gc
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    rng = np.random.default_rng(0)
    psfs = rng.random((1, 5, 5))
    x = rng.random((1, 512, 512)) + 0.1          # 2 MB results
    h = _lib.DeconvHandle(lib, psfs, x.shape[1:], precision=64)
    h.create_data(x, None, 3)
    a = h.get(_lib.TRUE_OBJECT)
    assert a.dtype == np.float64 and a.shape == x.shape and a.flags.c_contiguous and a.flags.writeable
    assert np.allclose(a, x, rtol=1e-14)
    addr = a.ctypes.data
    b = h.get(_lib.NOISELESS, 0)
    assert b.ctypes.data != addr                  # `a` is alive: not handed out twice
    keep = a[:, 10:20]                            # a view keeps the buffer alive
    del a
    gc.collect()
    c = h.get(_lib.NOISELESS, 0)
    assert c.ctypes.data != addr and np.allclose(keep, x[:, 10:20], rtol=1e-14)
    del keep
    gc.collect()
    d = h.get(_lib.NOISELESS, 0)
    assert d.ctypes.data == addr                  # recycled
    assert np.array_equal(d, b)
    h.close()


@pytest.mark.parametrize('shape', [(96, 128), (45, 50), (128, 75), (14, 128), (77, 91), (2048, 2048)])
def test_error_spectrum_on_device(shape):
    """record_iteration's log(1 + |fftshift(fft2(estimate - true_object))|) (ref:539-546)
    from the un-padded device transform: even / odd sides, the estimate in HBM or a host
    image; sides with a prime factor above 5 go through the direct transform (no host path)."""
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    rng = np.random.default_rng(3)
    psfs = rng.random((2, 5, 5))
    obj = rng.random((1,) + shape) + 0.1
    for precision, tol in ((64, 1e-12), (32, 2e-4)):   # fp32: bins near zero carry the transform's noise
        h = _lib.DeconvHandle(lib, psfs, shape, precision=precision)
        h.create_data(obj, 1e4 * obj.size, 5)
        h.iterate(2)
        est, true = h.get(_lib.ESTIMATE), h.get(_lib.TRUE_OBJECT)
        got = h.ft_error()
        assert got is not None
        want = np.log(1 + np.abs(np.fft.fftshift(np.fft.fftn(est - true, axes=(1, 2)), axes=(1, 2))))
        assert got.shape == want.shape
        assert np.abs(got - want).max() <= tol * np.abs(want).max()
        other = rng.random((1,) + shape) * true.mean()
        got = h.ft_error(other)
        want = np.log(1 + np.abs(np.fft.fftshift(np.fft.fftn(other - true, axes=(1, 2)), axes=(1, 2))))
        assert np.abs(got - want).max() <= tol * np.abs(want).max()
        h.iterate(1)        # the scratch image it used does not disturb the iteration state
        assert np.isfinite(h.get(_lib.ESTIMATE)).all()
        h.close()
