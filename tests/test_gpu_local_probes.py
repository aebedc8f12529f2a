"""Targeted probes of single CTAs and tiles on the GPU, with references computed without an FFT.

An impulse lattice: the output of H is a sum of shifted PSF copies, placed by slicing in fp64.
The lattice is staggered (every second lattice column shifted by one PSF height), so the
responses cover every image row, hence every row group and every tile, while each impulse keeps
a PSF-sized gap of exact zeros on all sides; more impulses sit on the four borders and corners.
H_t of this project convolves with the un-flipped PSFs, like the reference (oracle H_t), so its
reference is the same placement, summed over the orientations with a different weight per k.
Every pixel is checked with the local metrics of _local_error, and the exact-zero gaps must stay
at the transform's noise floor.

Stale state: on one handle, with the default graph replay, the lattice goes through H and H_t
before and after a random input and must come out bit for bit the same; and a Richardson-Lucy run
on the noisy measurements of one object after a run on another must match the oracle's run on
the second alone."""
import gc

import numpy as np
import pytest

import test_gpu_dispatch_parity as dp
import test_gpu_tiled_parity as tp
from _local_error import check_local, local_errors, unit, geometry
from oracle import line_sted_oracle as orc

pytestmark = pytest.mark.gpu

# Largest |output| in the exact-zero gaps of the lattice, over the largest |reference| of the
# same k, in units of eps * log2(Ly * Lx): 4x or more the worst measured on one NVIDIA B200
# (1000 W power limit), 0.33 (tiled_2x2_fp32 H) and 0.23 (plan2160d_fp64 H_t).
ZERO_BOUND = {32: 1.5, 64: 1.0}

# (handle kind, case): the fixed 2048 instances with complex and with centred real OTFs, fp64
# Plan2160d, generic columns with C = 1, generic rows with PR = 1, the orientation split of small
# frames over idle SMs, and a 2 x 2 grid of overlap-save tiles.
PROBES = {
    'fixed_2048_complex_otf_fp32': ('plain', dp.CASES['fixed_2048_asym107']),
    'fixed_2048_centred_otf_fp32': ('plain', dp.case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2))),
    'plan2160d_fp64': ('plain', dp.CASES['fp64_fig2_sub1']),
    'generic_C1_fp32': ('plain', dp.CASES['generic_fp32_C1_6075']),
    'generic_PR1_fp32': ('plain', dp.CASES['generic_fp32_PR1_7200']),
    'k_split_fp32': ('plain', dp.case((128, 128), 'asym107', 32, (192, 192, 4, 2), K=10)),
    'tiled_2x2_fp32': ('tiled', tp.CASES['w2160_asym21_fp32']),
}


def open_probe(name, monkeypatch):
    kind, c = PROBES[name]
    gc.collect()                        # k_split: handles of earlier tests must not count as live
    if kind == 'tiled':
        return tp.open_handle(c), c, tp.make_psfs(c.psf, c.K)
    return dp.open_handle(c, monkeypatch), c, dp.make_psfs(c.psf, c.K)


def lattice(shape, psf_shape):
    """Impulse positions: a staggered lattice of step twice the PSF size plus the borders."""
    (Ny, Nx), (ny, nx) = shape, psf_shape
    sy, sx = (ny - 1) // 2, (nx - 1) // 2
    pts = {(r, c) for j, c in enumerate(range(sx, Nx, 2 * nx))
           for r in range(sy + (j % 2) * ny, Ny, 2 * ny)}
    pts |= {(r, c) for r in (0, Ny // 2, Ny - 1) for c in (0, Nx // 2, Nx - 1)}
    return sorted(pts)


def place(pts, psf, shape):
    """sum of PSF copies, one per impulse, cropped like fftconvolve_same (fp64, no FFT)."""
    (Ny, Nx), (ny, nx) = shape, psf.shape
    full = np.zeros((Ny + ny - 1, Nx + nx - 1))
    for r, c in pts:
        full[r:r + ny, c:c + nx] += psf
    return full[(ny - 1) // 2:(ny - 1) // 2 + Ny, (nx - 1) // 2:(nx - 1) // 2 + Nx]


def zero_floor(got, want, gaps):
    """Largest |got| in the gaps over the largest |want|, per image."""
    got, want = got.reshape(want.shape), want
    return [np.abs(g[gaps]).max() / np.abs(w).max() for g, w in zip(got, want)] if gaps.any() else [0.0]


@pytest.mark.parametrize('name', sorted(PROBES))
def test_impulse_lattice_before_and_after_other_input(name, monkeypatch):
    h, c, psfs = open_probe(name, monkeypatch)
    try:
        info = h.info()
        pts = lattice(c.shape, psfs.shape[1:])
        x = np.zeros((1,) + c.shape)
        for r, col in pts:
            x[0, r, col] = 1.0
        w = 1.0 + np.arange(c.K)
        y = w[:, None, None] * x
        want_H = np.stack([place(pts, p, c.shape) for p in psfs])
        want_Ht = (w[:, None, None] * want_H).sum(0)[None]
        gaps = place(pts, np.ones(psfs.shape[1:]), c.shape) == 0
        H, Ht = h.H(x), h.Ht(y, False)
        rng = np.random.default_rng(5)          # another input through the same buffers
        h.H(rng.random((1,) + c.shape))
        h.Ht(rng.random((c.K,) + c.shape), False)
        H2, Ht2 = h.H(x), h.Ht(y, False)
        u = unit(c.precision, geometry(info))
        zero = {'H': zero_floor(H, want_H, gaps), 'Ht': zero_floor(Ht, want_Ht, gaps)}
        print('measured %s zero gaps (fp%d, %d impulses, %.0f%% of pixels): %s' % (
            name, c.precision, len(pts), 100 * gaps.mean(),
            ', '.join('%s %.2e = %.3g u' % (k, max(v), max(v) / u) for k, v in zero.items())))
        check_local([(name + ' lattice H', local_errors(H, want_H, info, c.precision)),
                     (name + ' lattice Ht', local_errors(Ht, want_Ht, info, c.precision))])
        for op, v in zero.items():
            k = int(np.argmax(v))
            assert v[k] <= ZERO_BOUND[c.precision] * u, (
                '%s %s: k = %d, exact-zero gaps: %.2e > %.2e' % (name, op, k, v[k], ZERO_BOUND[c.precision] * u))
        assert np.array_equal(H, H2), 'H of the lattice changed after another input'
        assert np.array_equal(Ht, Ht2), 'H_t of the lattice changed after another input'
    finally:
        h.close()


@pytest.mark.parametrize('name', sorted(PROBES))
def test_iterations_on_new_measurements_match_a_fresh_run(name, monkeypatch):
    from rescan_line_sted_b200 import _lib
    h, c, psfs = open_probe(name, monkeypatch)
    try:
        a = dp.make_object(c.shape, 'positive')
        b = np.random.default_rng(17).random((1,) + c.shape) + 0.1
        B = 100.0 * a.size
        o = orc.Deconvolver([p[None] for p in psfs])
        o.create_data_from_object(b, total_brightness=B, random_seed=9)
        o.iterate(), o.iterate()
        h.create_data(a, B, 3)
        for _ in range(3):
            h.iterate(1)
        for k in range(c.K):
            h.set(_lib.NOISY, k, o.noisy_measurement[k])
        h.set_option('reset_estimate', 1)
        h.iterate(1)
        h.iterate(1)
        got = h.get(_lib.ESTIMATE)
        assert h.info().iterations_done == 2
        check_local([(name + ' object B after A, iter2',
                      local_errors(got, o.estimate, h.info(), c.precision, estimate=True))])
    finally:
        h.close()
