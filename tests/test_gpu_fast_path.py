"""The compile-time-planned kernels (L = 2160) against the generic kernels
and the oracle at a size the oracle finishes in seconds."""
import numpy as np
import pytest

from oracle import line_sted_oracle as orc

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    return np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b))


@pytest.mark.parametrize('precision,tol', [(64, 1e-12), (32, 1e-5)])
@pytest.mark.parametrize('shape', [(2100, 2100), (2048, 2101), (2089, 2048)])
def test_fast_path_matches_oracle_and_generic(precision, tol, shape):
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    rng = np.random.default_rng(0)
    psfs = rng.random((2, 9, 11))
    Ny, Nx = shape
    x = rng.random((1, Ny, Nx))
    y = rng.random((2, Ny, Nx))
    o = orc.Deconvolver([p[None] for p in psfs])
    Hx = np.concatenate(o.H(x))
    Hty = o.H_t([v[None] for v in y], normalize=False)
    h = _lib.DeconvHandle(lib, psfs, shape, precision=precision)
    info = h.info()
    assert (info.Ly, info.Lx) == (2160, 2160)
    assert rel_l2(h.H(x), Hx) < tol
    assert rel_l2(h.Ht(y, False), Hty) < tol
    h.create_data(x, 1e9, 0)
    noisy = [h.get(_lib.NOISY, k) for k in range(2)]
    h.iterate(2)
    o.create_data_from_object(x, 1e9, 0)
    o.noisy_measurement = noisy
    o.iterate(), o.iterate()
    assert rel_l2(h.get(_lib.ESTIMATE), o.estimate) < 10 * tol
    if precision == 32:   # the generic kernels fit in shared memory for fp32 only
        g = _lib.DeconvHandle(lib, psfs, shape, precision=precision)
        g.set_option('fast_path', 0)
        assert rel_l2(g.H(x), Hx) < tol
        g.create_data(x, 1e9, 0)
        for k in range(2):
            g.set(_lib.NOISY, k, noisy[k])
        g.iterate(2)
        assert rel_l2(g.get(_lib.ESTIMATE), h.get(_lib.ESTIMATE)) < 10 * tol
        g.close()
    h.close()


@pytest.mark.parametrize('shape,K', [((64, 2048), 2), ((1184, 2048), 2), ((801, 2048), 3), ((2048, 2048), 4)])
def test_tensor_map_row_staging_is_bit_identical(shape, K):
    """ROW_MID / ROW_FINAL move their spectrum chunks by tensor-map TMA (option `row_tma`,
    default on); the arithmetic is the same, so the estimates must agree bit for bit with the
    per-thread LDG/STG kernels.  Sizes on both sides of two full waves of row CTAs and of a
    20 MB spectrum array, an odd row count, and the last orientation (whose chunks end the
    allocation)."""
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    rng = np.random.default_rng(3)
    psfs = rng.random((K, 3, 21))
    x = rng.random((1,) + shape) + 0.1
    est = {}
    for tma in (0, 1, 2):   # 2: also the two-buffer ROW_MID (measurement rows read in place)
        h = _lib.DeconvHandle(lib, psfs, shape, precision=32)
        assert h.info().Lx == 2160          # the rows run the 2160 plan, where row_tma applies
        h.set_option('row_tma', tma)
        h.create_data(x, 1e6 * x.size, 1)
        h.iterate(3)
        est[tma] = h.get(_lib.ESTIMATE)
        h.close()
    assert np.isfinite(est[1]).all() and est[1].min() > 0
    assert np.array_equal(est[0], est[1])
    assert np.array_equal(est[0], est[2])


@pytest.mark.gpu
@pytest.mark.parametrize('shape,K', [((2048, 64), 2), ((2048, 2048), 3), ((2101, 1030), 2)])
def test_sub_block_column_ctas_are_bit_identical(shape, K):
    """Column kernels on centred real OTFs as sub-block CTAs (2 of 4 columns, two CTAs per
    SM; option `col_sub`, default on) against the whole-block CTAs: bit-identical estimates."""
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    rng = np.random.default_rng(8)
    half = rng.random((K, 10, 21))
    psfs = np.concatenate([half, rng.random((K, 1, 21)), half[:, ::-1, ::-1]], axis=1)
    psfs[:, 10, :] = 0.5 * (psfs[:, 10, :] + psfs[:, 10, ::-1])
    x = rng.random((1,) + shape) + 0.1
    est = {}
    for sub in (0, 1):
        h = _lib.DeconvHandle(lib, psfs, shape, precision=32)
        assert h.info().Ly == 2160          # the columns run the 2160 plan, where col_sub applies
        h.set_option('col_sub', sub)
        h.create_data(x, 1e6 * x.size, 1)
        h.iterate(3)
        est[sub] = h.get(_lib.ESTIMATE)
        h.close()
    assert np.isfinite(est[1]).all() and est[1].min() > 0
    assert np.array_equal(est[0], est[1])


@pytest.mark.gpu
@pytest.mark.parametrize('shape,K,precision', [((128, 128), 4, 32), ((128, 160), 3, 64),
                                               ((2048, 2048), 2, 32)])
def test_graph_replay_of_the_iteration_is_bit_identical(shape, K, precision):
    """The steady RL iteration replayed as a captured CUDA graph (option `graph`, default on)
    against four plain launches: same kernels, same arguments -> identical bits; new data,
    a reset estimate, an option change and mixed iterate(1) / iterate(n) calls in between."""
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    rng = np.random.default_rng(11)
    psfs = rng.random((K, 9, 11))
    x = rng.random((1,) + shape) + 0.1
    est = {}
    for graph in (0, 1):
        h = _lib.DeconvHandle(lib, psfs, shape, precision=precision)
        h.set_option('graph', graph)
        h.create_data(x, 1e6 * x.size, 1)
        for _ in range(3):
            h.iterate(1)
        h.iterate(4)
        a = h.get(_lib.ESTIMATE)
        h.set_option('exact_clip', 1)
        h.iterate(2)
        h.set_option('exact_clip', 0)
        h.iterate(3)
        b = h.get(_lib.ESTIMATE)
        h.create_data(x[:, ::-1].copy(), 2e6 * x.size, 2)      # new data, estimate restarts
        h.iterate(5)
        est[graph] = (a, b, h.get(_lib.ESTIMATE))
        h.close()
    for u, v in zip(est[0], est[1]):
        assert np.isfinite(v).all() and v.min() > 0
        assert np.array_equal(u, v)


@pytest.mark.gpu
@pytest.mark.parametrize('K', [2, 4, 10])
def test_orientations_of_small_frames_over_idle_sms_are_bit_identical(K):
    """Generic col_h on the reference's own frame size (128^2, 107^2 PSFs): the K orientations
    of a column block spread over the idle SMs (option `k_split`, default on) against one CTA
    per block: same arithmetic per orientation -> identical bits."""
    from rescan_line_sted_b200 import _lib
    lib = _lib.get()
    rng = np.random.default_rng(17)
    psfs = rng.random((K, 107, 107))
    x = rng.random((1, 128, 128)) + 0.1
    est = {}
    for split in (0, 1):
        h = _lib.DeconvHandle(lib, psfs, (128, 128), precision=32)
        h.set_option('k_split', split)
        h.create_data(x, 1e6 * x.size, 1)
        h.iterate(5)
        est[split] = (h.get(_lib.ESTIMATE), h.get(_lib.NOISELESS, K - 1))
        h.close()
    for u, v in zip(est[0], est[1]):
        assert np.isfinite(v).all() and v.min() >= 0
        assert np.array_equal(u, v)
