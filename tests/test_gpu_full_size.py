"""BASELINE config 4 at its full size (2048^2 object, 16 orientations of the figure-2
rescan PSF, fp32) through the C ABI: direct parity with the oracle where the oracle
finishes in seconds, and size-independent properties of the operators for the rest
(impulse response, linearity, adjointness for point-symmetric PSFs, Richardson-Lucy
fixed point, Poisson moments).  Tolerance of BASELINE.json: rel-L2 <= 1e-5 in fp32."""
import os

import numpy as np
import pytest

import bench
from _local_error import check_local, local_errors
from oracle import line_sted_oracle as orc

pytestmark = pytest.mark.gpu
N, K, TOL = 2048, 16, 1e-5


def rel_l2(a, b):
    return np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b))


@pytest.fixture(scope='module')
def setup(golden_dir):
    from rescan_line_sted_b200 import _lib, line_sted_tools as st, orientations
    base = np.load(os.path.join(golden_dir, 'fig2_2p0x_lr.npz'))['base_psf']
    psfs = orientations.line_orientation_psfs(base, K, bench.EMISSION_2P0X_LR)
    ref = orc.orientation_psfs(base, K, bench.EMISSION_2P0X_LR)
    for p, r in zip(psfs, ref):
        assert rel_l2(p, r) < 1e-12
    h = _lib.DeconvHandle(_lib.get(), st._stack_psfs(psfs), (N, N), precision=32)
    info = h.info()
    assert (info.Ly, info.Lx) == (2160, 2160)
    yield h, psfs, _lib
    h.close()


def test_forward_model_against_oracle_on_two_orientations(setup):
    h, psfs, _lib = setup
    obj = bench.synthetic_object(N)
    h.create_data(obj, bench.total_brightness(N), 0)
    scaled = obj * (bench.total_brightness(N) / obj.sum())
    assert rel_l2(h.get(_lib.TRUE_OBJECT), scaled) < 1e-6
    for k in (0, 7):
        want = np.clip(orc.fftconvolve_same(scaled, psfs[k]), 0, None)
        assert rel_l2(h.get(_lib.NOISELESS, k), want) < TOL, k


def test_impulse_response_is_the_psf(setup):
    h, psfs, _lib = setup
    x = np.zeros((1, N, N))
    spots = [(1000, 1100), (53, 53), (N - 54, 70), (0, 0), (N - 1, N - 1)]
    for (r, c) in spots:
        x[0, r, c] = 1.0
    out = h.H(x)
    n = psfs[0].shape[-1]
    s = (n - 1) // 2
    for k in range(K):
        want = np.zeros((N + 2 * s, N + 2 * s))
        for (r, c) in spots:
            want[r:r + n, c:c + n] += psfs[k][0]
        want = want[s:s + N, s:s + N]
        assert np.abs(out[k] - want).max() <= 2e-6 * psfs[k].max(), k


def test_linearity_and_adjointness(setup):
    h, psfs, _lib = setup
    rng = np.random.default_rng(1)
    x, z = rng.random((1, N, N)), rng.random((1, N, N))
    Hx, Hz = h.H(x), h.H(z)
    assert rel_l2(h.H(2.0 * x + 0.5 * z), 2.0 * Hx + 0.5 * Hz) < TOL
    # H_t convolves with the un-flipped PSFs (ref:586); it is the adjoint of H because the
    # PSFs are point-symmetric about their centre
    for p in psfs:
        assert np.abs(p - p[:, ::-1, ::-1]).max() < 1e-12 * p.max()
    y = rng.random((K, N, N))
    lhs = float(np.sum(Hx.astype(np.float64) * y))
    rhs = float(np.sum(x * h.Ht(y, False)))
    assert abs(lhs - rhs) <= TOL * abs(lhs)
    ones = h.Ht(np.ones((K, N, N)), False)
    assert rel_l2(h.get(_lib.NORMALIZATION), ones) < TOL


def test_richardson_lucy_fixed_point_and_one_oracle_iteration(setup):
    h, psfs, _lib = setup
    rng = np.random.default_rng(2)
    x = rng.random((1, N, N)) + 0.5
    h.create_data(x, None, 0)
    for k in range(K):                       # noise-free measurement: x is a fixed point
        h.set(_lib.NOISY, k, h.get(_lib.NOISELESS, k))
    h.set(_lib.ESTIMATE, 0, x)
    h.iterate(3)
    assert rel_l2(h.get(_lib.ESTIMATE), x) < 10 * TOL
    # one full RL iteration from the flat start against the oracle (2K = 32 convolutions)
    noisy = [h.get(_lib.NOISELESS, k) * (1.0 + 0.1 * rng.random((1, N, N))) for k in range(K)]
    for k in range(K):
        h.set(_lib.NOISY, k, noisy[k])
    h.set(_lib.ESTIMATE, 0, np.ones((1, N, N)))
    h.iterate(1)
    import scipy.fft
    o = orc.Deconvolver(psfs)
    o.noisy_measurement = noisy
    with scipy.fft.set_workers(os.cpu_count()):
        o.iterate()
    assert rel_l2(h.get(_lib.ESTIMATE), o.estimate) < 10 * TOL


def test_poisson_moments_at_full_size(setup):
    h, psfs, _lib = setup
    obj = bench.synthetic_object(N)
    h.create_data(obj, bench.total_brightness(N), 5)
    for k in (0, 9, 15):
        lam = h.get(_lib.NOISELESS, k)[0, 64:-64, 64:-64].astype(np.float64)
        cnt = h.get(_lib.NOISY, k)[0, 64:-64, 64:-64].astype(np.float64)
        z = (cnt - lam) / np.sqrt(np.maximum(lam, 1.0))
        n = z.size
        # fp32 storage rounds counts above 2^24 to multiples of 2; moments are unaffected
        assert abs(z.mean()) < 5 / np.sqrt(n) + 1e-3
        assert abs(z.var() - 1.0) < 5 * np.sqrt(2.0 / n) + 2e-3


# ---------------------------------------------------------------------------
# Round 2: the benched configuration itself (2048^2, K = 16, figure-2 PSFs -> centred real
# OTFs, 2160 fast path) on the objects of SURVEY.md 8d, in both H_t clip orders, and the
# drift over the 64 iterations the headline runs.
# ---------------------------------------------------------------------------
# Tolerance per RL iteration count (fp32 engine against fp64 results on identical inputs):
# one pass through the operators is the 1e-5 of BASELINE.json; every further multiplicative
# update adds its own fp32 round-off, so the budget grows with the iteration count
# (SURVEY.md section 7, hard part 8).  Measured values are printed and written to
# gpurun_out/parity_r02.json by these tests.
TOL_ITER = {1: 1e-5, 2: 1e-5, 8: 1e-5, 64: 2e-5}   # measured on B200: 2e-7, 3e-7, 9e-7, 7e-6 (profiles/r02_parity_measured.json)
_measured = {}


def _record(name, value):
    import json
    _measured[name] = float(value)
    print('measured %s = %.3e' % (name, value))
    try:
        os.makedirs(os.path.join(os.path.dirname(__file__), '..', 'gpurun_out'), exist_ok=True)
        with open(os.path.join(os.path.dirname(__file__), '..', 'gpurun_out', 'parity_r02.json'), 'w') as f:
            json.dump(_measured, f, indent=1, sort_keys=True)
    except OSError:
        pass


def object_O2():
    return np.random.default_rng(2048).random((1, N, N))


def object_O3():
    """Sparse beads of SURVEY.md 8d: zeros with 1.0 at N*N/1024 random pixels."""
    obj = np.zeros((1, N, N))
    idx = np.random.default_rng(7).integers(0, N, (N * N // 1024, 2))
    obj[0, idx[:, 0], idx[:, 1]] = 1.0
    return obj


def test_forward_model_against_oracle_on_all_orientations(setup):
    h, psfs, _lib = setup
    import scipy.fft
    obj = bench.synthetic_object(N)
    h.create_data(obj, bench.total_brightness(N), 0)
    scaled = obj * (bench.total_brightness(N) / obj.sum())
    with scipy.fft.set_workers(os.cpu_count()):
        want = np.concatenate([np.clip(orc.fftconvolve_same(scaled, psfs[k]), 0, None) for k in range(K)])
    got = np.concatenate([h.get(_lib.NOISELESS, k) for k in range(K)])
    worst = max(rel_l2(got[k], want[k]) for k in range(K))
    _record('forward_O1_all16_fp32', worst)
    check_local([('forward O1 noiseless', local_errors(got, want, h.info(), 32))])
    assert worst < TOL


@pytest.mark.parametrize('name', ['O2_random', 'O3_sparse_beads'])
def test_objects_O2_O3_create_inject_iterate_both_clip_orders(setup, name):
    """create_data -> inject the oracle's noise field -> 2 iterations, against the oracle, with
    the Fourier-domain H_t sum (default) and with the reference's clip-per-term order."""
    h, psfs, _lib = setup
    import scipy.fft
    obj = object_O2() if name.startswith('O2') else object_O3()
    B = bench.total_brightness(N)
    o = orc.Deconvolver(psfs)
    with scipy.fft.set_workers(os.cpu_count()):
        o.create_data_from_object(obj, total_brightness=B, random_seed=0)
        h.set_option('exact_clip', 0)
        h.create_data(obj, B, 0)
        got = np.concatenate([h.get(_lib.NOISELESS, k) for k in range(K)])
        worst = max(rel_l2(got[k], o.noiseless_measurement[k]) for k in range(K))
        _record('forward_%s_fp32' % name, worst)
        check_local([('forward %s noiseless' % name,
                      local_errors(got, np.concatenate(o.noiseless_measurement), h.info(), 32))])
        assert worst < TOL
        est = {}
        for n_it in (1, 2):
            o.iterate()
            est[n_it] = o.estimate.copy()
    for exact in (0, 1):
        h.set_option('exact_clip', exact)
        h.set_option('forget_normalization', 1)
        h.create_data(obj, B, 0)
        for k in range(K):
            h.set(_lib.NOISY, k, o.noisy_measurement[k])
        for n_it in (1, 2):
            h.iterate(1)
            got = h.get(_lib.ESTIMATE)
            assert np.isfinite(got).all()
            err = rel_l2(got, est[n_it])
            _record('estimate_%s_iter%d_exact_clip%d_fp32' % (name, n_it, exact), err)
            check_local([('%s iter%d exact_clip %d' % (name, n_it, exact),
                          local_errors(got, est[n_it], h.info(), 32, estimate=True))])
            assert err < TOL_ITER[n_it], (name, exact, n_it, err)
    h.set_option('exact_clip', 0)
    h.set_option('forget_normalization', 1)


def test_sixty_four_iteration_drift_fp32_vs_fp64(setup):
    """The headline runs 64 fp32 iterations: same PSFs, object, injected noise in an fp64 handle
    (itself pinned against the oracle at 1e-12, tests below and test_gpu_fast_path) as the
    yardstick, checked at 1, 8 and 64 iterations against the written per-count tolerance."""
    h, psfs, _lib = setup
    from rescan_line_sted_b200 import line_sted_tools as st
    obj = bench.synthetic_object(N)
    B = bench.total_brightness(N)
    d = _lib.DeconvHandle(_lib.get(), st._stack_psfs(psfs), (N, N), precision=64)
    d.create_data(obj, B, 11)
    h.create_data(obj, B, 11)
    for k in range(K):
        h.set(_lib.NOISY, k, d.get(_lib.NOISY, k))
    done = 0
    for n_it in (1, 8, 64):
        h.iterate(n_it - done), d.iterate(n_it - done)
        done = n_it
        err = rel_l2(h.get(_lib.ESTIMATE), d.get(_lib.ESTIMATE))
        _record('drift_O1_iter%d_fp32_vs_fp64' % n_it, err)
        assert err < TOL_ITER[n_it], (n_it, err)
    d.close()


def test_sixty_four_iterations_against_the_oracle_at_512(golden_dir):
    """Where the oracle can afford 64 iterations (512^2, K = 4): fp64 engine <= 1e-10 and fp32
    engine within the per-count tolerance of the ORACLE's estimate."""
    from rescan_line_sted_b200 import _lib, line_sted_tools as st
    import scipy.fft
    n, k4 = 512, 4
    base = np.load(os.path.join(golden_dir, 'fig2_2p0x_lr.npz'))['base_psf']
    psfs = orc.orientation_psfs(base, k4, bench.EMISSION_2P0X_LR)
    obj = bench.synthetic_object(n)
    B = bench.total_brightness(n)
    o = orc.Deconvolver(psfs)
    hs = {p: _lib.DeconvHandle(_lib.get(), st._stack_psfs(psfs), (n, n), precision=p) for p in (32, 64)}
    with scipy.fft.set_workers(os.cpu_count()):
        o.create_data_from_object(obj, total_brightness=B, random_seed=3)
        for p, hh in hs.items():
            hh.create_data(obj, B, 3)
            for k in range(k4):
                hh.set(_lib.NOISY, k, o.noisy_measurement[k])
        done = 0
        for n_it in (1, 8, 64):
            for _ in range(n_it - done):
                o.iterate()
            for hh in hs.values():
                hh.iterate(n_it - done)
            done = n_it
            e64 = rel_l2(hs[64].get(_lib.ESTIMATE), o.estimate)
            e32 = rel_l2(hs[32].get(_lib.ESTIMATE), o.estimate)
            _record('oracle512_iter%d_fp64' % n_it, e64)
            _record('oracle512_iter%d_fp32' % n_it, e32)
            assert e64 < 1e-10, (n_it, e64)
            assert e32 < TOL_ITER[n_it], (n_it, e32)
    for hh in hs.values():
        hh.close()


def test_dark_background_at_full_size_fp32(setup):
    """Zero-background object (a few beads, the rest of the 2048^2 frame dark): the fp32
    forward model is FFT round-off there, half of it clipped to 0 -> expected == 0.  Pinned
    decision: ratio 0 for such pixels, the estimate stays finite and non-zero (the reference
    would divide by zero; see tests/test_robustness.py)."""
    h, psfs, _lib = setup
    obj = np.zeros((1, N, N))
    idx = np.random.default_rng(5).integers(200, N - 200, (40, 2))
    obj[0, idx[:, 0], idx[:, 1]] = 1.0
    h.create_data(obj, 1e9, 2)
    noiseless = np.stack([h.get(_lib.NOISELESS, k) for k in range(K)])
    assert (noiseless == 0).mean() > 0.2          # the clip really produces exact zeros
    h.iterate(12)
    est = h.get(_lib.ESTIMATE)
    assert np.isfinite(est).all() and est.min() >= 0 and est.sum() > 0
    # the light is still at the beads: >= 90 % of the estimate within 30 px of a bead
    mask = np.zeros((N, N), bool)
    for (r, c) in idx:
        mask[max(0, r - 30):r + 31, max(0, c - 30):c + 31] = True
    assert est[0][mask].sum() > 0.9 * est.sum()
