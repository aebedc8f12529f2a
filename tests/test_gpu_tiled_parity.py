"""The overlap-save tiled engine (tiled.h + the window kernels of ew_bodies.cuh) on the GPU,
against the fp64 oracle, across tile grids, PSF shapes and tile FFT lengths.

Inside a window the engine runs the convolution with Ny = Nx = Ly = Lx = W and complex OTFs,
a geometry that never occurs untiled; the window kernels carry the negative window origins,
the ragged last tile, the asymmetric halos of even PSFs and the guarded ratio.  Each case is one
row of data and asserts the `info()` that selects its path first (tile grid, interior size,
transform lengths, columns and row pairs per CTA), so that a planner change fails the case
instead of quietly testing another path.  Every quantity is checked twice: rel-L2 over the whole
image, and the largest single-pixel error (relative to the largest value) on the strips around
the tile seams, the last tile row and column and the image border, where one wrong row would
otherwise be diluted by the rest of the image."""
import os
import zlib
from collections import namedtuple
from functools import lru_cache

import numpy as np
import pytest

import bench
from _local_error import check_local, local_errors
from oracle import line_sted_oracle as orc

pytestmark = pytest.mark.gpu

TOL = {32: (1e-5, 1e-4), 64: (1e-12, 1e-11)}     # (operators, after RL iterations)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'fig2_2p0x_lr.npz')

Case = namedtuple('Case', 'shape psf K precision tile_len options info obj')


def case(shape, psf, precision, info, K=2, tile_len=2160, options=(), obj='positive'):
    return Case(shape, psf, K, precision, tile_len, tuple(options), info, obj)


# info = (tiles_y, tiles_x, tile_out_y, tile_out_x, Ly, Lx, cols_per_cta, row_pairs_per_cta);
# tile_out = W - (PSF side - 1).  PSF kinds: 'asym<n>' random n x n, 'asym<ny>x<nx>' random
# ny x nx, 'fig2' the figure-2 rescan PSFs (107 x 107, point-symmetric), 'one' 1 x 1.
CASES = {
    # 2 x 2 grids of 2160 windows: complex OTFs on the 2160 plan along both axes
    'w2160_asym21_fp32': case((2200, 2300), 'asym21', 32, (2, 2, 2140, 2140, 2160, 2160, 4, 2), K=3),
    'w2160_asym21_fp64': case((2200, 2300), 'asym21', 64, (2, 2, 2140, 2140, 2160, 2160, 2, 2), K=3),
    'w2160_asym9x11_fp32': case((2200, 2300), 'asym9x11', 32, (2, 2, 2152, 2150, 2160, 2160, 4, 2)),
    'w2160_asym9x11_fp64': case((2200, 2300), 'asym9x11', 64, (2, 2, 2152, 2150, 2160, 2160, 2, 2)),
    # crop offset 53 wrapping inside Ny = Ly windows
    'w2160_asym107_fp32': case((2200, 2300), 'asym107', 32, (2, 2, 2054, 2054, 2160, 2160, 4, 2)),
    # the config-5 PSFs: point-symmetric, yet complex OTFs inside windows
    'w2160_fig2_fp32': case((2200, 2300), 'fig2', 32, (2, 2, 2054, 2054, 2160, 2160, 4, 2), K=4),
    'w2160_fig2_fp64': case((2200, 2300), 'fig2', 64, (2, 2, 2054, 2054, 2160, 2160, 2, 2), K=4),
    # even PSF sides: first interior row / column ny-1-sy != sy
    'w2160_even_10x12_fp64': case((2200, 2300), 'asym10x12', 64, (2, 2, 2151, 2149, 2160, 2160, 2, 2)),
    # 1 x 3 grid, a different halo per axis
    'w2160_rect_9x31_1x3': case((1500, 4300), 'asym9x31', 32, (1, 3, 2152, 2130, 2160, 2160, 4, 2)),
    # 3 x 1 grid whose last tile is one row tall (2 * 2140 + 1)
    'w2160_3x1_thin_last': case((4281, 700), 'asym21', 64, (3, 1, 2140, 2140, 2160, 2160, 2, 2)),
    # no halo: the whole window is interior
    'w2160_one_pixel_psf': case((2200, 2300), 'one', 32, (2, 2, 2160, 2160, 2160, 2160, 4, 2)),
    # per-term clip inside windows
    'w2160_exact_clip_fp64': case((2200, 2300), 'asym21', 64, (2, 2, 2140, 2140, 2160, 2160, 2, 2),
                                  K=3, options=[('exact_clip', 1)]),
    # generic kernels and row options inside 2160 windows (set on the backend the tiles share)
    'w2160_fast_path0': case((2200, 2300), 'asym21', 32, (2, 2, 2140, 2140, 2160, 2160, 4, 2),
                             K=3, options=[('fast_path', 0)]),
    'w2160_row_tma0': case((2200, 2300), 'asym21', 32, (2, 2, 2140, 2140, 2160, 2160, 4, 2),
                           K=3, options=[('row_tma', 0)]),
    'w2160_row_plan2': case((2200, 2300), 'asym21', 32, (2, 2, 2140, 2140, 2160, 2160, 4, 2),
                            K=3, options=[('row_plan2', 1)]),
    # generic window lengths; radix schedules 16*4, 16*4*3, 9*8*3, 16*5*3, 9*8*5*3
    'generic_w64_fp32': case((150, 170), 'asym9x11', 32, (3, 4, 56, 54, 64, 64, 4, 2), tile_len=64),
    'generic_w64_fp64_even': case((47, 201), 'asym10x12', 64, (1, 4, 55, 53, 64, 64, 2, 2), tile_len=64),
    'generic_w192_fp32_even': case((600, 1000), 'asym10x12', 32, (4, 6, 183, 181, 192, 192, 4, 2),
                                   tile_len=192),
    'generic_w216_fp64': case((600, 1000), 'asym9x11', 64, (3, 5, 208, 206, 216, 216, 2, 2), tile_len=216),
    'generic_w240_fp32': case((600, 1000), 'asym9x11', 32, (3, 5, 232, 230, 240, 240, 4, 2), tile_len=240),
    'generic_w1080_fp64': case((2200, 2300), 'asym9x11', 64, (3, 3, 1072, 1070, 1080, 1080, 2, 2),
                               tile_len=1080),
    # the automatic switch to tiles (column transform too long for shared memory)
    'auto_fp64_4500x64': case((4500, 64), 'asym9', 64, (3, 1, 2152, 2152, 2160, 2160, 2, 2), tile_len=0),
    'auto_fp32_9000x64': case((9000, 64), 'asym21', 32, (5, 1, 2140, 2140, 2160, 2160, 4, 2), tile_len=0),
    # beads on a zero background: the ratio is 0 where the expected value is 0
    'dark_fp32': case((2200, 2300), 'fig2', 32, (2, 2, 2054, 2054, 2160, 2160, 4, 2), obj='dark'),
}


def oracle_key(name):
    c = CASES[name]
    return (c.shape, c.psf, c.K, c.obj, name)


def rel_l2(a, b):
    return np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b))


@lru_cache(maxsize=None)
def make_psfs(kind, K):
    rng = np.random.default_rng(zlib.crc32(kind.encode()) + K)
    if kind == 'fig2':
        from rescan_line_sted_b200 import orientations
        base = np.load(GOLDEN)['base_psf']
        return np.stack([p[0] for p in orientations.line_orientation_psfs(base, K, bench.EMISSION_2P0X_LR)])
    if kind == 'one':
        return rng.random((K, 1, 1)) + 0.5
    sides = [int(v) for v in kind[4:].split('x')]
    return rng.random((K, sides[0], sides[-1]))


def make_object(shape, obj):
    rng = np.random.default_rng(shape[0] * 7919 + shape[1])
    if obj == 'positive':
        return rng.random((1,) + shape) + 0.1
    x = np.zeros((1,) + shape)          # 'dark': beads on a zero background
    idx = rng.integers(0, min(shape), (max(8, shape[0] * shape[1] // 4096), 2))
    x[0, idx[:, 0], idx[:, 1]] = 1.0
    return x


@lru_cache(maxsize=2)
def oracle_results(shape, psf, K, obj):
    """float64 oracle: H of the object, H_t of K random images (unnormalised and normalised),
    the normalisation, the noiseless and noisy fields of create_data and the estimates after
    one and two RL iterations from that noisy field."""
    import scipy.fft
    psfs = make_psfs(psf, K)
    x = make_object(shape, obj)
    y = np.random.default_rng(1).random((K,) + shape)
    o = orc.Deconvolver([p[None] for p in psfs])
    B = 100.0 * x.size
    with scipy.fft.set_workers(os.cpu_count()), np.errstate(divide='ignore', invalid='ignore'):
        r = {'x': x, 'y': y, 'B': B, 'H': np.concatenate(o.H(x))}
        ylist = [v[None] for v in y]
        r['Ht'] = o.H_t(ylist, normalize=False)
        r['Ht_norm'] = o.H_t(ylist)
        r['norm'] = o.H_t_normalization
        o.create_data_from_object(x, total_brightness=B, random_seed=3)
        r['noiseless'] = np.concatenate(o.noiseless_measurement)
        r['noisy'] = o.noisy_measurement
        r['est'] = []
        for _ in range(2):
            o.iterate()
            r['est'].append(o.estimate.copy())
    assert all(np.isfinite(e).all() for e in r['est'])
    return r


def seam_mask(shape, info, psf_shape):
    """Strips of +-(PSF size) around every tile seam, the last tile row and column, and a
    PSF-wide border of the image."""
    ny, nx = psf_shape
    m = np.zeros(shape, bool)
    for t in range(1, info.tiles_y):
        m[max(t * info.tile_out_y - ny, 0):t * info.tile_out_y + ny] = True
    for t in range(1, info.tiles_x):
        m[:, max(t * info.tile_out_x - nx, 0):t * info.tile_out_x + nx] = True
    m[(info.tiles_y - 1) * info.tile_out_y:] = True
    m[:, (info.tiles_x - 1) * info.tile_out_x:] = True
    m[:ny] = m[-ny:] = True
    m[:, :nx] = m[:, -nx:] = True
    return m


def errors(got, want, mask):
    """(rel-L2 over the image, largest error on `mask` relative to the largest value)."""
    got, want = np.asarray(got).reshape(-1, *mask.shape), np.asarray(want).reshape(-1, *mask.shape)
    seam = np.abs(got - want)[:, mask].max() / np.abs(want).max()
    return rel_l2(got, want), seam


def lib():
    from rescan_line_sted_b200 import _lib
    return _lib.get()


def open_handle(c):
    from rescan_line_sted_b200 import _lib
    h = _lib.DeconvHandle(lib(), make_psfs(c.psf, c.K), c.shape, precision=c.precision,
                          tile_fft_len=c.tile_len)
    info = h.info()
    got = (info.tiles_y, info.tiles_x, info.tile_out_y, info.tile_out_x,
           info.Ly, info.Lx, info.cols_per_cta, info.row_pairs_per_cta)
    assert got == c.info
    for name, value in c.options:
        h.set_option(name, value)
    return h


def check_against_oracle(h, c, label):
    from rescan_line_sted_b200 import _lib
    r = oracle_results(c.shape, c.psf, c.K, c.obj)
    info = h.info()
    mask = seam_mask(c.shape, info, make_psfs(c.psf, c.K).shape[1:])
    H, Ht = h.H(r['x']), h.Ht(r['y'], False)
    err = {'H': errors(H, r['H'], mask),
           'Ht': errors(Ht, r['Ht'], mask),
           'Ht_norm': errors(h.Ht(r['y'], True), r['Ht_norm'], mask),
           'norm': errors(h.get(_lib.NORMALIZATION), r['norm'], mask)}
    local = [(label + ' H', local_errors(H, r['H'], info, c.precision)),
             (label + ' Ht', local_errors(Ht, r['Ht'], info, c.precision))]
    h.create_data(r['x'], r['B'], 3)
    noiseless = np.concatenate([h.get(_lib.NOISELESS, k) for k in range(c.K)])
    err['noiseless'] = errors(noiseless, r['noiseless'], mask)
    local.append((label + ' noiseless', local_errors(noiseless, r['noiseless'], info, c.precision)))
    for k in range(c.K):
        h.set(_lib.NOISY, k, r['noisy'][k])
    for n in (1, 2):
        h.iterate(1)
        got = h.get(_lib.ESTIMATE)
        assert np.isfinite(got).all() and got.min() >= 0
        err['iter%d' % n] = errors(got, r['est'][n - 1], mask)
        local.append(('%s iter%d' % (label, n),
                      local_errors(got, r['est'][n - 1], info, c.precision, estimate=True)))
    assert h.info().iterations_done == 2
    print('measured %s (fp%d): %s' % (label, c.precision, ', '.join(
        '%s %.2e/%.2e' % (name, l2, seam) for name, (l2, seam) in err.items())))
    check_local(local)
    tol_op, tol_it = TOL[c.precision]
    for name, (l2, seam) in err.items():
        tol = tol_it if name.startswith('iter') else tol_op
        assert l2 < tol, (label, name, 'rel-L2', l2)
        assert seam < tol, (label, name, 'seams', seam)
    return got


@pytest.mark.parametrize('name', sorted(CASES, key=oracle_key))
def test_tiled_path_against_oracle(name):
    c = CASES[name]
    h = open_handle(c)
    try:
        check_against_oracle(h, c, name)
    finally:
        h.close()


@pytest.mark.parametrize('shape,psf,precision,Ly', [((4090, 64), 'asym9', 64, 4096),
                                                    ((8990, 64), 'asym21', 32, 9000)])
def test_largest_untiled_columns_stay_untiled(shape, psf, precision, Ly):
    """The other side of the automatic switch of auto_fp64_4500x64 / auto_fp32_9000x64: the
    longest column transforms that still fit shared memory (one column per CTA) stay untiled."""
    from rescan_line_sted_b200 import _lib
    h = _lib.DeconvHandle(lib(), make_psfs(psf, 2), shape, precision=precision)
    info = h.info()
    h.close()
    assert (info.tiles_y, info.tiles_x, info.Ly, info.cols_per_cta) == (1, 1, Ly, 1)


# ---------------------------------------------------------------------------
# Error spectrum, state protocol, tiled against untiled
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('precision,tol', [(64, 1e-12), (32, 2e-4)])
def test_error_spectrum_on_tiled_handle(precision, tol):
    """record_iteration's log(1 + |fftshift(fft2(image - true_object))|) of a tiled object: the
    direct transform over 2200 x 2300 pixels.  It uses the host-transfer buffer as scratch; the
    next iteration must not depend on it."""
    from rescan_line_sted_b200 import _lib
    c = CASES['w2160_asym21_fp%d' % precision]
    h = open_handle(c)
    try:
        x = make_object(c.shape, 'positive')
        h.create_data(x, 100.0 * x.size, 5)
        h.iterate(2)
        est, true = h.get(_lib.ESTIMATE), h.get(_lib.TRUE_OBJECT)
        got = h.ft_error()
        want = np.log(1 + np.abs(np.fft.fftshift(np.fft.fftn(est - true, axes=(1, 2)), axes=(1, 2))))
        err = np.abs(got - want).max() / np.abs(want).max()
        other = np.random.default_rng(4).random((1,) + c.shape) * true.mean()
        got = h.ft_error(other)
        want = np.log(1 + np.abs(np.fft.fftshift(np.fft.fftn(other - true, axes=(1, 2)), axes=(1, 2))))
        err_other = np.abs(got - want).max() / np.abs(want).max()
        print('measured ft_error tiled fp%d: estimate %.2e, host image %.2e' % (precision, err, err_other))
        assert err <= tol and err_other <= tol
        h.iterate(1)
        after = h.get(_lib.ESTIMATE)
        h.set(_lib.ESTIMATE, 0, est)      # est holds the engine's values exactly
        h.iterate(1)
        assert np.array_equal(h.get(_lib.ESTIMATE), after)
    finally:
        h.close()


def signed_psfs():
    """PSFs with negative lobes, one of negative sum: clipping each term of H_t differs from
    clipping their sum."""
    p = np.random.default_rng(8).random((3, 9, 11))
    p[1] -= 0.7
    return p


def test_state_protocol_on_tiled_handle():
    """iterate(n) against n calls of iterate(1), reset_estimate, set(ESTIMATE) (the estimate's
    halo is fresh), set(NORMALIZATION), and exact_clip dropping the cached normalisation, on a
    3 x 3 grid of 256-point windows (fp64)."""
    import scipy.signal
    from rescan_line_sted_b200 import _lib
    shape, W = (600, 700), 256
    psfs = make_psfs('asym9x11', 3)
    r = oracle_results(shape, 'asym9x11', 3, 'positive')
    tol_op, tol_it = TOL[64]
    h = _lib.DeconvHandle(lib(), psfs, shape, precision=64, tile_fft_len=W)
    try:
        info = h.info()
        assert (info.tiles_y, info.tiles_x, info.Ly) == (3, 3, W)
        h.create_data(r['x'], r['B'], 3)
        for k in range(3):
            h.set(_lib.NOISY, k, r['noisy'][k])
        h.iterate(2)
        assert h.info().iterations_done == 2
        two = h.get(_lib.ESTIMATE)
        assert rel_l2(two, r['est'][1]) < tol_it
        h.set_option('reset_estimate', 1)
        assert h.info().iterations_done == 0
        h.iterate(1)
        assert h.info().iterations_done == 1
        assert rel_l2(h.get(_lib.ESTIMATE), r['est'][0]) < tol_it   # restarted from ones
        h.iterate(1)
        assert np.array_equal(h.get(_lib.ESTIMATE), two)

        rng = np.random.default_rng(6)
        e = rng.random((1,) + shape) + 0.5
        n = rng.random((1,) + shape) + 1.0
        for norm in (None, n):
            o = orc.Deconvolver([p[None] for p in psfs])
            o.noisy_measurement = r['noisy']
            o.estimate, o.num_iterations = e.copy(), 1
            if norm is not None:
                o.H_t_normalization = norm
                h.set(_lib.NORMALIZATION, 0, norm)
            o.iterate()
            h.set(_lib.ESTIMATE, 0, e)
            h.iterate(1)
            err = rel_l2(h.get(_lib.ESTIMATE), o.estimate)
            print('measured set(ESTIMATE)%s + iterate: %.2e' % (
                '' if norm is None else ' + set(NORMALIZATION)', err))
            assert err < tol_it

        h.close()
        h = _lib.DeconvHandle(lib(), signed_psfs(), shape, precision=64, tile_fft_len=W)
        ones = np.ones(shape)
        terms = [scipy.signal.fftconvolve(ones, p, mode='same') for p in signed_psfs()]
        summed = np.clip(sum(terms), 0, None)
        per_term = sum(np.clip(t, 0, None) for t in terms)
        assert rel_l2(summed, per_term) > 1e-3
        assert rel_l2(h.get(_lib.NORMALIZATION)[0], summed) < tol_op
        h.set_option('exact_clip', 1)
        assert rel_l2(h.get(_lib.NORMALIZATION)[0], per_term) < tol_op
        h.set_option('exact_clip', 0)
        assert rel_l2(h.get(_lib.NORMALIZATION)[0], summed) < tol_op
    finally:
        h.close()


@pytest.mark.parametrize('precision', [32, 64])
def test_tiled_equals_untiled_on_device(precision):
    """An object that fits one plain transform, once through 3 x 3 windows of 256 points and once
    untiled: the same operators, the same noise field (fp64: pixel for pixel; the Philox
    counters are the global pixel index) and the same iterations."""
    from rescan_line_sted_b200 import _lib
    shape = (600, 700)
    psfs = make_psfs('asym9x11', 3)
    r = oracle_results(shape, 'asym9x11', 3, 'positive')
    tol_op, tol_it = TOL[precision]
    tiled = _lib.DeconvHandle(lib(), psfs, shape, precision=precision, tile_fft_len=256)
    plain = _lib.DeconvHandle(lib(), psfs, shape, precision=precision)
    try:
        assert (tiled.info().tiles_y, tiled.info().tiles_x) == (3, 3)
        assert (plain.info().tiles_y, plain.info().tiles_x) == (1, 1)
        err = {'H': rel_l2(tiled.H(r['x']), plain.H(r['x'])),
               'Ht': rel_l2(tiled.Ht(r['y'], False), plain.Ht(r['y'], False)),
               'Ht_norm': rel_l2(tiled.Ht(r['y'], True), plain.Ht(r['y'], True))}
        tiled.create_data(r['x'], r['B'], 9)
        plain.create_data(r['x'], r['B'], 9)
        err['noiseless'] = max(rel_l2(tiled.get(_lib.NOISELESS, k), plain.get(_lib.NOISELESS, k))
                               for k in range(3))
        for k in range(3):
            noisy = plain.get(_lib.NOISY, k)
            if precision == 64:
                assert np.array_equal(tiled.get(_lib.NOISY, k), noisy)
            tiled.set(_lib.NOISY, k, noisy)
        tiled.iterate(2)
        plain.iterate(2)
        err['iter2'] = rel_l2(tiled.get(_lib.ESTIMATE), plain.get(_lib.ESTIMATE))
        print('measured tiled vs untiled (fp%d): %s' % (
            precision, ', '.join('%s %.2e' % kv for kv in err.items())))
        for name, e in err.items():
            assert e < (tol_it if name.startswith('iter') else tol_op), (name, e)
    finally:
        tiled.close()
        plain.close()


def test_simulate_uses_the_uploaded_object():
    """upload_object stages the object that every later simulate() draws from, however many
    reads, writes and operators run in between (a frame loop uploads once)."""
    from rescan_line_sted_b200 import _lib
    c = CASES['w2160_asym9x11_fp64']
    r = oracle_results(c.shape, c.psf, c.K, c.obj)
    h = open_handle(c)
    try:
        h.upload_object(np.ascontiguousarray(r['x']))
        h.get(_lib.ESTIMATE)
        h.ft_error(r['x'])
        h.simulate(r['B'], 3)
        got = np.concatenate([h.get(_lib.NOISELESS, k) for k in range(c.K)])
        assert rel_l2(got, r['noiseless']) < TOL[64][0]
    finally:
        h.close()
