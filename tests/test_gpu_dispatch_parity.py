"""Every kernel path the engine dispatches to on the GPU, against the fp64 oracle, and the GPU
noise field against the textbook sampler, pixel for pixel.

The engine picks its kernels per axis and per launch (lsted_api.cu: launch_row / launch_col):
the compile-time 2160 plan when the transform length is 2160 and the column geometry has the
plan's C, else the generic Stockham kernels with C = 4, 2, 1 columns and PR = 2, 1 row pairs per
CTA; fixed-geometry instances for 2048-wide images (RowGeom2048 / ColGeom2048 with complex OTFs,
RowGeom2048c / ColGeom2048c with centred real OTFs of point-symmetric PSFs); tensor-map row
staging, the two-pass and dual row plans, sub-block column CTAs and the split of the
orientations over idle SMs.  Each case below is one row of data and asserts the `info()` that
selects its path first, so that a planner change fails the case instead of quietly testing
another path."""
import gc
import os
import zlib
from collections import namedtuple
from functools import lru_cache

import numpy as np
import pytest

import bench
from _local_error import check_local, local_errors
from _poisson_replay import assert_field
from oracle import line_sted_oracle as orc

pytestmark = pytest.mark.gpu

TOL = {32: (1e-5, 1e-4), 64: (1e-12, 1e-11)}     # (operators, after two RL iterations)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'fig2_2p0x_lr.npz')

Case = namedtuple('Case', 'shape psf K precision options env info obj')


def case(shape, psf, precision, info, K=2, options=(), env=(), obj='positive'):
    return Case(shape, psf, K, precision, tuple(options), tuple(env), info, obj)


# info = (Ly, Lx, cols_per_cta, row_pairs_per_cta).  PSF kinds: 'asym<n>' random n x n,
# 'sym<n>' its point-symmetric part (centred real OTFs where the columns run the 2160 plan),
# 'fig2' the figure-2 rescan PSFs (107 x 107, point-symmetric), 'one' 1 x 1.
CASES = {
    # 2160 rows + generic columns; row_tma 2 falls back to 1 where Nx * 4 % 16 != 0
    'fastrows_gencols_tma0': case((64, 2048), 'asym21', 32, (75, 2160, 4, 2), options=[('row_tma', 0)]),
    'fastrows_gencols_tma1': case((64, 2048), 'asym21', 32, (75, 2160, 4, 2), options=[('row_tma', 1)]),
    'fastrows_gencols_tma2': case((64, 2048), 'asym21', 32, (75, 2160, 4, 2), options=[('row_tma', 2)]),
    'fastrows_gencols_odd_2049': case((801, 2049), 'asym21', 32, (864, 2160, 4, 2)),
    'fastrows_gencols_fp64': case((64, 2048), 'asym21', 64, (75, 2160, 2, 2)),
    # generic rows + 2160 columns on centred real OTFs
    'genrows_fastcols_2048c_sub0': case((2048, 64), 'sym21', 32, (2160, 75, 4, 2), options=[('col_sub', 0)]),
    'genrows_fastcols_2048c_sub1': case((2048, 64), 'sym21', 32, (2160, 75, 4, 2), options=[('col_sub', 1)]),
    'genrows_fastcols_runtime_fp32': case((2101, 40), 'sym21', 32, (2160, 50, 4, 2)),
    'genrows_fastcols_runtime_fp64': case((2101, 40), 'sym21', 64, (2160, 50, 2, 2)),
    # fixed-geometry instances with complex OTFs
    'fixed_2048_asym107': case((2048, 2048), 'asym107', 32, (2160, 2160, 4, 2)),
    'fixed_2048_fig2_complex_otf': case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2),
                                        env=[('LSTED_REAL_OTF', '0')]),
    # fp64 2160 plan on centred real OTFs (Plan2160d, one-column sub-block CTAs)
    'fp64_fig2_sub0': case((2048, 2048), 'fig2', 64, (2160, 2160, 2, 2), options=[('col_sub', 0)]),
    'fp64_fig2_sub1': case((2048, 2048), 'fig2', 64, (2160, 2160, 2, 2), options=[('col_sub', 1)]),
    'fp64_fig2_exact_clip': case((2048, 2048), 'fig2', 64, (2160, 2160, 2, 2), options=[('exact_clip', 1)]),
    'fp64_fig2_runtime_dark': case((2047, 1999), 'fig2', 64, (2160, 2160, 2, 2), obj='dark'),
    # row-kernel options on the headline geometry
    'fig2_row_plan2': case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2), options=[('row_plan2', 1)]),
    'fig2_row_dual': case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2), options=[('row_dual', 1)]),
    'fig2_prefetch0': case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2), options=[('prefetch', 0)]),
    # Lx = 2160 but generic rows: the column geometry has C != the plan's C
    'lx2160_genrows_fp32_C2': case((2300, 2048), 'asym21', 32, (2400, 2160, 2, 2)),
    'lx2160_genrows_fp64_C1': case((2500, 2048), 'asym21', 64, (2560, 2160, 1, 2)),
    # generic fallbacks and long transforms
    'generic_fp32_C2': case((2300, 8), 'asym21', 32, (2400, 24, 2, 2)),
    'generic_fp32_C1_6075': case((6000, 96), 'asym21', 32, (6075, 108, 1, 2)),
    'generic_fp32_PR1_7200': case((96, 7000), 'asym21', 32, (108, 7200, 4, 1)),
    'generic_fp64_C1': case((2300, 8), 'asym21', 64, (2400, 24, 1, 2)),
    'generic_fp64_PR1_3375': case((4, 3300), 'asym21', 64, (24, 3375, 2, 1)),
    'generic_fp32_3125': case((8, 3125), 'one', 32, (8, 3125, 4, 2)),
    'generic_fp64_3125': case((8, 3125), 'one', 64, (8, 3125, 2, 2)),
    # schedules ending in radix 2, 4, 8 after the 16s: 32 = 16*2, 64 = 16*4, 128 = 16*8
    'radix_tail_fp32_32x64': case((28, 60), 'asym9', 32, (32, 64, 4, 2)),
    'radix_tail_fp32_128': case((124, 124), 'asym9', 32, (128, 128, 4, 2)),
    'radix_tail_fp64_64x32': case((60, 28), 'asym9', 64, (64, 32, 2, 2)),
    'radix_tail_fp64_128': case((124, 124), 'asym9', 64, (128, 128, 2, 2)),
    # generic kernels at L = 2160 (fast path off), complex and centred OTFs
    'fast_path0_2160_asym': case((2048, 2048), 'asym21', 32, (2160, 2160, 4, 2), options=[('fast_path', 0)]),
    'fast_path0_2160_fig2': case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2), options=[('fast_path', 0)]),
}


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
    n = int(kind[4:] if kind.startswith('asym') else kind[3:])
    p = rng.random((K, n, n))
    return 0.5 * (p + p[:, ::-1, ::-1]) if kind.startswith('sym') else p


def make_object(shape, obj):
    rng = np.random.default_rng(shape[0] * 7919 + shape[1])
    if obj == 'positive':
        return rng.random((1,) + shape) + 0.1
    x = np.zeros((1,) + shape)          # 'dark': beads on a zero background
    idx = rng.integers(0, min(shape), (max(8, shape[0] * shape[1] // 4096), 2))
    x[0, idx[:, 0], idx[:, 1]] = 1.0
    return x


@lru_cache(maxsize=3)
def oracle_results(shape, psf, K, obj):
    """H, H_t (unnormalised), the noiseless and noisy fields of create_data and the estimates
    after one and two RL iterations, in float64 by the oracle."""
    import scipy.fft
    psfs = make_psfs(psf, K)
    x = make_object(shape, obj)
    y = np.random.default_rng(1).random((K,) + shape)
    o = orc.Deconvolver([p[None] for p in psfs])
    B = 100.0 * x.size
    with scipy.fft.set_workers(os.cpu_count()):
        Hx = np.concatenate(o.H(x))
        Hty = o.H_t([v[None] for v in y], normalize=False)
        o.create_data_from_object(x, total_brightness=B, random_seed=3)
        est = []
        for _ in range(2):
            o.iterate()
            est.append(o.estimate.copy())
    return x, y, B, Hx, Hty, o.noiseless_measurement, o.noisy_measurement, est


def open_handle(c, monkeypatch):
    from rescan_line_sted_b200 import _lib
    for name, value in c.env:           # read by the backend when the handle is created
        monkeypatch.setenv(name, value)
    h = _lib.DeconvHandle(_lib.get(), make_psfs(c.psf, c.K), c.shape, precision=c.precision)
    for name, _ in c.env:
        monkeypatch.delenv(name)
    info = h.info()
    assert (info.Ly, info.Lx, info.cols_per_cta, info.row_pairs_per_cta) == c.info
    for name, value in c.options:
        h.set_option(name, value)
    return h


def check_against_oracle(h, c, label):
    from rescan_line_sted_b200 import _lib
    x, y, B, Hx, Hty, noiseless, noisy, est = oracle_results(c.shape, c.psf, c.K, c.obj)
    tol_op, tol_it = TOL[c.precision]
    info = h.info()
    got = {'H': h.H(x), 'Ht': h.Ht(y, False)}
    h.create_data(x, B, 3)
    got['noiseless'] = np.concatenate([h.get(_lib.NOISELESS, k) for k in range(c.K)])
    for k in range(c.K):
        h.set(_lib.NOISY, k, noisy[k])
    for n in (1, 2):
        h.iterate(1)
        got['iter%d' % n] = h.get(_lib.ESTIMATE)
        assert np.isfinite(got['iter%d' % n]).all()
    want = {'H': Hx, 'Ht': Hty, 'noiseless': np.concatenate(noiseless),
            'iter1': est[0], 'iter2': est[1]}
    err = {'H': rel_l2(got['H'], Hx), 'Ht': rel_l2(got['Ht'], Hty),
           'noiseless': max(rel_l2(got['noiseless'][k], noiseless[k]) for k in range(c.K)),
           'iter1': rel_l2(got['iter1'], est[0]), 'iter2': rel_l2(got['iter2'], est[1])}
    print('measured %s (fp%d): %s' % (label, c.precision,
                                      ', '.join('%s %.2e' % kv for kv in err.items())))
    local = [('%s %s' % (label, name), local_errors(got[name], want[name], info, c.precision,
                                                   estimate=name.startswith('iter')))
             for name in want]
    check_local(local)
    for name, e in err.items():
        assert e < (tol_it if name.startswith('iter') else tol_op), (label, name, e)
    return got['iter2']


@pytest.mark.parametrize('name', sorted(CASES))
def test_dispatch_path_against_oracle(name, monkeypatch):
    c = CASES[name]
    h = open_handle(c, monkeypatch)
    try:
        check_against_oracle(h, c, name)
    finally:
        h.close()


def test_orientation_split_against_oracle_with_and_without_other_handles(monkeypatch):
    """The reference's frame size (128^2, K = 10, 107^2 PSFs): COL_H spreads the orientations
    of a column block over idle SMs only while at most two handles are live.  Both launch
    shapes against the oracle, and bit-identical to each other."""
    from rescan_line_sted_b200 import _lib
    c = case((128, 128), 'asym107', 32, (192, 192, 4, 2), K=10)
    gc.collect()                        # handles of earlier tests must not count as live
    h = open_handle(c, monkeypatch)
    alone = check_against_oracle(h, c, 'k_split_alone')
    h.close()
    others = [_lib.DeconvHandle(_lib.get(), np.ones((1, 3, 3)), (16, 16)) for _ in range(2)]
    h = open_handle(c, monkeypatch)
    crowded = check_against_oracle(h, c, 'k_split_three_handles')
    h.close()
    for o in others:
        o.close()
    assert np.array_equal(alone, crowded)


# ---------------------------------------------------------------------------
# The noise field of create_data, pixel for pixel
# ---------------------------------------------------------------------------
def noise_object(shape, psfs):
    """Object whose noiseless images hold exact zeros (a dark stretch wider than the PSFs,
    clipped FFT round-off), lambda in (0, 10), lambda in [10, 1e4] and lambda ~ 2e7 (above 2^24,
    where fp32 storage rounds the counts), in bands across the columns."""
    Ny, Nx = shape
    rng = np.random.default_rng(Nx)
    gain = psfs.sum(axis=(1, 2)).min()
    x = np.empty((1, Ny, Nx))
    edges = np.linspace(0, Nx, 5).astype(int)
    bands = [(0.0, 0.0), (0.5, 8.0), (20.0, 9e3), (1.9e7, 2.1e7)]
    for (lo, hi), a, b in zip(bands, edges[:-1], edges[1:]):
        x[0, :, a:b] = rng.uniform(lo, hi, (Ny, b - a)) / gain
    return x


NOISE_CASES = {
    'fp32_fast_RowGeom2048c': case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2)),
    'fp32_fast_RowGeom2048': case((2048, 2048), 'asym107', 32, (2160, 2160, 4, 2)),
    'fp32_fast_runtime_odd_rows': case((801, 2049), 'asym21', 32, (864, 2160, 4, 2)),
    'fp32_row_plan2': case((512, 2048), 'fig2', 32, (576, 2160, 4, 2), options=[('row_plan2', 1)]),
    'fp64_Plan2160d': case((2048, 2048), 'fig2', 64, (2160, 2160, 2, 2)),
    'fp32_generic_rows': case((300, 500), 'asym21', 32, (320, 512, 4, 2)),
    'fp64_generic_rows': case((300, 500), 'asym21', 64, (320, 512, 2, 2)),
}


@pytest.mark.parametrize('name', sorted(NOISE_CASES))
def test_noise_field_is_the_textbook_field(name, monkeypatch):
    from rescan_line_sted_b200 import _lib
    c = NOISE_CASES[name]
    h = open_handle(c, monkeypatch)
    seed = 0x2545F4914F6CDD1D
    try:
        h.create_data(noise_object(c.shape, make_psfs(c.psf, c.K)), None, seed)
        check_noise_field(h, c.K, seed, c.precision)
    finally:
        h.close()


def check_noise_field(h, K, seed, precision):
    from rescan_line_sted_b200 import _lib
    for k in range(K):
        lam = h.get(_lib.NOISELESS, k)
        assert (lam == 0).any() and ((lam > 0) & (lam < 10)).any()
        assert ((lam >= 10) & (lam <= 1e4)).any() and (lam > 2 ** 24).any()
        assert_field(h.get(_lib.NOISY, k), lam, seed, k, np.float32 if precision == 32 else np.float64)


def test_tiled_noise_field_is_the_textbook_field():
    """The overlap-save tiled engine draws the noise per tile (WIN_SIMULATE) with the global
    pixel index: the same field."""
    from rescan_line_sted_b200 import _lib
    psfs = make_psfs('asym21', 2)
    h = _lib.DeconvHandle(_lib.get(), psfs, (2200, 2300), precision=64, tile_fft_len=2160)
    seed = 77
    try:
        info = h.info()
        assert (info.tiles_y, info.tiles_x) == (2, 2) and (info.Ly, info.Lx) == (2160, 2160)
        h.create_data(noise_object((2200, 2300), psfs), None, seed)
        check_noise_field(h, 2, seed, 64)
    finally:
        h.close()
