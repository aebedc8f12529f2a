"""Tiled engine on the GPU at config-5 scale (8192^2 tiles, fp64) through exact
local checks: a linear convolution is local, so any patch of the tiled result
must equal the oracle's convolution of the patch plus its halo.  The tile grids,
PSF shapes and window lengths against the whole-image oracle are in
test_gpu_tiled_parity.py."""
import numpy as np
import pytest

from oracle import line_sted_oracle as orc

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    return np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b))


def test_config5_scale_local_exactness():
    """Config 5 as BASELINE.json states it: 8192^2 object, 32 orientations of the 107^2
    figure-2 rescan PSF, fp64, automatic tiling (4 x 4 tiles of 2054^2).  A linear convolution
    is local, so patches of the tiled results must equal the oracle run on the patch plus its
    halo: the forward model on patch + 53 px, one full RL iteration (H, ratio, H_t,
    normalisation, update) on patch + 106 px with the device's own Poisson field injected.
    Patches sit inside a tile, across tile seams (2054, 4108, 6162) and at image corners."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    from rescan_line_sted_b200 import _lib, line_sted_tools as st
    N, K, n = 8192, 32, 107
    base = st.psf_report('line', verbose=False, **bench.FIG2_2P0X_LR)['psfs']['rescan_sted']
    psf_list = bench.orientation_psfs(base, K)
    psfs = st._stack_psfs(psf_list)
    x = np.random.default_rng(2).random((1, N, N)) + 0.05
    h = _lib.DeconvHandle(_lib.get(), psfs, (N, N), precision=64)     # tiles automatically
    info = h.info()
    assert (info.tiles_y, info.tiles_x) == (4, 4) and info.tile_out_y == 2054 and info.K == K
    brightness = bench.total_brightness(N)
    h.create_data(x, brightness, 11)
    scaled = x * (brightness / x.sum())
    half, size = n // 2, 96
    patches = ((0, 0), (2054 - 40, 2054 - 50), (4108 - 10, 6162 - 80), (N - size, N - size), (3000, 5000))

    def grown(py, px, halo):
        return max(py - halo, 0), min(py + size + halo, N), max(px - halo, 0), min(px + size + halo, N)

    noisy_sub = {p: [] for p in patches}
    worst_fwd = 0.0
    for k in range(K):
        nl = h.get(_lib.NOISELESS, k)
        noisy = h.get(_lib.NOISY, k)
        for (py, px) in patches:
            y0, y1, x0, x1 = grown(py, px, half)
            o = orc.Deconvolver([psf_list[k]])
            want = o.H(scaled[:, y0:y1, x0:x1])[0][:, py - y0:py - y0 + size, px - x0:px - x0 + size]
            worst_fwd = max(worst_fwd, rel_l2(nl[:, py:py + size, px:px + size], want))
            y0, y1, x0, x1 = grown(py, px, 2 * half)
            noisy_sub[(py, px)].append(noisy[:, y0:y1, x0:x1].copy())
        if k == 0:   # Poisson field: integer counts, right mean
            counts = noisy - 1e-9
            assert np.abs(counts - np.round(counts)).max() < 1e-6
            assert abs((counts - nl).mean()) < 5 * np.sqrt(nl.mean() / nl.size)
    assert worst_fwd < 1e-12, worst_fwd
    h.iterate(1)
    est = h.get(_lib.ESTIMATE)
    assert np.isfinite(est).all() and est.min() >= 0
    worst_it = 0.0
    for (py, px) in patches:
        y0, y1, x0, x1 = grown(py, px, 2 * half)
        o = orc.Deconvolver(psf_list)
        o.noisy_measurement = noisy_sub[(py, px)]
        o.iterate()
        want = o.estimate[:, py - y0:py - y0 + size, px - x0:px - x0 + size]
        worst_it = max(worst_it, rel_l2(est[:, py:py + size, px:px + size], want))
    assert worst_it < 1e-11, worst_it
    h.close()
