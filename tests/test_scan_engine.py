"""Figure-3 scan-position engine (SURVEY.md 8f row 2; line_sted_figure_3.py:76-273, :382-409).

 * the oracle (oracle/scan_oracle.py, scipy calls like the reference) against frames captured
   from the UNMODIFIED reference function (tests/golden/fig3_frames.npz, make_golden_fig3.py);
 * the engine (rescan_line_sted_b200/scan_engine.py -> liblsted.so) against those frames and
   against the oracle: on the CPU replay of the kernel functors here, on the GPU under -m gpu;
 * the scan-position counts of the reference's own table (appendix.html:325-369).
fp64 throughout.  Tolerance: every display plane within 1e-11 of its maximum (they are scaled
to [0, 1]); sums of planes within 1e-11 relative; counters exact."""
import json
import os

import numpy as np
import pytest

import emul_support
from oracle import scan_oracle
from rescan_line_sted_b200 import _lib

KEYS = ('excitation', 'glow', 'inst_sig', 'cum_sig', 'new_sig', 'reconstruction')
TOL = 1e-11


@pytest.fixture(scope='module')
def golden(golden_dir):
    return (np.load(os.path.join(golden_dir, 'fig3_frames.npz')),
            json.load(open(os.path.join(golden_dir, 'fig3_frames.json'))))


def lines_object(crop, tile=1):
    """test_object_lines.tif / 255 + 1e-6 like line_sted_figure_3.py:42, centre crop.  The 8-bit
    128^2 image the golden frames were captured on is stored in tests/golden/fig3_object_lines.npz."""
    here = os.path.dirname(os.path.abspath(__file__))
    u8 = np.load(os.path.join(here, 'golden', 'fig3_object_lines.npz'))['object_u8']
    obj = u8 / 255 + 1e-6
    lo = (128 - crop) // 2
    return np.tile(np.ascontiguousarray(obj[:, lo:lo + crop, lo:lo + crop]), (1, tile, tile))


def run_case(sim, meta):
    obj = lines_object(meta['crop'])
    frames = []

    def record(filename, *a):
        rot = int(os.path.basename(filename).split('deg_')[0].split('_')[-1])
        frames.append(dict(rot=rot, which_pos=int(filename[-10:-4]), arrays=[np.array(x) for x in a[:7]],
                           pulses_delivered=a[7], camera_exposures=a[8]))
    out = sim(obj, meta['imaging_type'], meta['psf_width'], meta['R'], meta['num_orientations'],
              meta['pulses_per_position'], meta['pad'], comparison_name='case',
              generate_figure=record, verbose=False)
    return out, frames


def check_against_golden(frames, name, golden):
    g, meta = golden
    m = meta[name]
    assert len(frames) == m['num_frames']
    sums = g[name + '/sums']
    compared = 0
    for i, (f, want) in enumerate(zip(frames, m['frames'])):
        assert [f['rot'], f['which_pos'], f['pulses_delivered'], f['camera_exposures']] == want
        for j, k in enumerate(KEYS):
            a = f['arrays'][j + 1]
            assert a.shape == (m['crop'], m['crop']) and a.dtype == np.float64
            assert abs(a.sum() - sums[i, j + 1, 0]) <= TOL * max(abs(sums[i, j + 1, 0]), 1.0), (name, i, k)
            assert abs(a.max() - sums[i, j + 1, 1]) <= TOL, (name, i, k)
            key = '%s/%03d/%06d/%s' % (name, f['rot'], f['which_pos'], k)
            if key in g.files:
                assert np.abs(a - g[key]).max() <= TOL, key
                compared += 1
        assert np.abs(f['arrays'][0].sum() - sums[i, 0, 0]) <= TOL * sums[i, 0, 0]
    assert compared >= 6


SMALL = ['small_descan_point', 'small_multipoint', 'small_descan_line', 'small_rescan_line',
         'small_rescan_line_R1', 'small_rescan_line_R3']
FULL = ['fig3_descan_line', 'fig3_rescan_line', 'fig3_multipoint']


def oracle_sim(obj, typ, width, R, n_or, pulses, pad, comparison_name, generate_figure, verbose):
    out = scan_oracle.simulate_imaging(obj, typ, width, R, n_or, pulses, pad)
    objd = np.pad(obj, ((0, 0), (pad, pad), (pad, pad)), 'constant')
    for f in out['frames']:
        generate_figure('x_%03ideg_case_%06i.svg' % (f['rot'], f['which_pos']),
                        objd[0, pad:-pad, pad:-pad] / objd.max(), f['excitation'], f['glow'],
                        f['inst_sig'], f['cum_sig'], f['new_sig'], f['reconstruction'],
                        f['pulses_delivered'], f['camera_exposures'])
    return out


@pytest.mark.parametrize('name', ['small_multipoint', 'small_descan_line', 'small_rescan_line_R1'])
def test_oracle_reproduces_reference_frames(name, golden):
    """The oracle is pinned: bit-for-bit the frames of the unmodified reference."""
    _, frames = run_case(oracle_sim, golden[1][name])
    check_against_golden(frames, name, golden)
    g, _ = golden
    for f in frames:
        for j, k in enumerate(KEYS):
            key = '%s/%03d/%06d/%s' % (name, f['rot'], f['which_pos'], k)
            if key in g.files:
                assert np.array_equal(f['arrays'][j + 1], g[key])


def engine():
    from rescan_line_sted_b200 import scan_engine
    return scan_engine


@pytest.fixture()
def emulated(monkeypatch):
    monkeypatch.setattr(_lib, '_library', emul_support.emulator_library())
    return engine()


@pytest.mark.parametrize('name', SMALL)
def test_engine_on_cpu_replay_against_reference_frames(name, golden, emulated):
    out, frames = run_case(emulated.simulate_imaging, golden[1][name])
    check_against_golden(frames, name, golden)


def check_helpers(se):
    from scipy import ndimage as ndi
    import warnings
    rng = np.random.default_rng(5)
    x = rng.random((1, 41, 53))
    for angle in (0, 30, 60, 90, 120, -45, 200.5):
        assert np.abs(se.rotate(x, angle) - scan_oracle.rotate(x, angle)).max() < 1e-12, angle
    x2 = rng.random((2, 81, 95))           # corners leave the edge-padded source
    for angle in (45, 17):
        ref = np.clip(ndi.rotate(x2, angle, axes=(1, 2), mode='nearest', reshape=False), 0, 1.1 * x2.max())
        assert np.abs(se.rotate(x2, angle) - ref).max() < 1e-12
    for s in ((0, 3, 0), (0, -7, 5), (0, 2.5, -1.25), (0, 60, 0)):
        assert np.abs(se.shift(x, s) - scan_oracle.shift(x, s)).max() < 1e-12, s
    for f in (0.5, 0.2, 0.1, 1 / 3):
        assert np.abs(se.scale_y(x, f) - scan_oracle.scale_y(x, f)).max() < 1e-12, f
    # lines of 160 samples and more take the blocked prefilter (warm-up windows instead of a walk
    # along the whole line): same numbers
    x3 = rng.random((1, 200, 170))
    assert np.abs(se.rotate(x3, 33.0) - scan_oracle.rotate(x3, 33.0)).max() < 1e-12
    assert np.abs(se.shift(x3, (0, 3.5, -2.25)) - scan_oracle.shift(x3, (0, 3.5, -2.25))).max() < 1e-12
    assert np.abs(se.scale_y(x3, 0.2) - scan_oracle.scale_y(x3, 0.2)).max() < 1e-12
    spike = np.zeros((1, 230, 161)); spike[0, 0, 0] = spike[0, -1, -1] = spike[0, 100, 80] = 1.0
    assert np.abs(se.rotate(spike, 10.0) - scan_oracle.rotate(spike, 10.0)).max() < 1e-13
    assert np.abs(se.shift(spike, (0, 0.5, 0.5)) - scan_oracle.shift(spike, (0, 0.5, 0.5))).max() < 1e-13
    for sigma, trunc in ((4.2, 4), ((0, 2.5, 0), 8), ((0, 3.1, 3.1), 8), (30.0, 4)):
        ref = ndi.gaussian_filter(x, sigma, truncate=trunc)
        assert np.abs(se.gaussian_filter(x, sigma, truncate=trunc) - ref).max() < 1e-13, sigma


def test_helpers_on_cpu_replay(emulated):
    check_helpers(emulated)


def test_scan_position_counts_of_the_reference_table(emulated):
    """appendix.html:325-369: scan positions of every method, R in {1, 2, 3}, 1x1 and 2x2 fields
    of view of the 128^2 objects, psf_width 25 (line_sted_figure_3.py:40-63).  The table prints
    131 line positions for R = 3, 2x2 -- inconsistent with its own point entry (16641 = 129^2)
    and with the script, which gives 129 = len(arange(-128, 129, 2)); 129 is pinned here."""
    table = {(1, 1): (484, 36, 22), (1, 2): (1849, 36, 43), (2, 1): (1849, 144, 43),
             (2, 2): (7396, 144, 86), (3, 1): (4225, 324, 65), (3, 2): (16641, 324, 129)}
    for (R, fov), (point, multi, line) in table.items():
        shape = (1, 128 * fov, 128 * fov)
        assert len(emulated.scan_plan(shape, 'descan_point', 25, R)[1]) == point
        assert len(emulated.scan_plan(shape, 'nondescan_multipoint', 25, R)[1]) == multi
        assert len(emulated.scan_plan(shape, 'descan_line', 25, R)[1]) == line
        assert len(emulated.scan_plan(shape, 'rescan_line', 25, R)[1]) == line


def test_chunked_scan_equals_one_pass(emulated, golden):
    """Positions processed in chunks (bounded device memory) give the same numbers."""
    meta = golden[1]['small_rescan_line']
    obj = lines_object(meta['crop'])
    padded = np.pad(obj, ((0, 0), (meta['pad'],) * 2, (meta['pad'],) * 2), 'constant')
    res = []
    for chunk_bytes in (0, 3 * 8 * padded.size * 5):      # everything at once / 5 positions a time
        h = emulated.ScanHandle('rescan_line', obj.shape, meta['pad'], meta['psf_width'], meta['R'],
                                chunk_bytes=chunk_bytes)
        keep = emulated.frames_drawn(len(h.positions))
        mx, recon, cum = h.run(padded, 60.0, keep)
        fr = h.frames(3, 4, [1, 2, 3, 4, 5, 6], 60.0)
        res.append((mx, recon, cum, fr))
        h.close()
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a, b)


def test_argument_checks(emulated):
    obj = np.ones((1, 16, 16))
    with pytest.raises(AssertionError):
        emulated.simulate_imaging(obj[0], 'rescan_line', 8, 2, 1, 1, 4, verbose=False)
    with pytest.raises(AssertionError):
        emulated.simulate_imaging(obj, 'confocal', 8, 2, 1, 1, 4, verbose=False)
    with pytest.raises(AssertionError):
        emulated.simulate_imaging(obj, 'rescan_line', 8, 0.5, 1, 1, 4, verbose=False)
    with pytest.raises(AssertionError):
        emulated.simulate_imaging(obj, 'rescan_line', 8, 2, 1, 1, 0, verbose=False)
    h = emulated.ScanHandle('descan_line', obj.shape, 4, 8, 2)
    with pytest.raises(RuntimeError, match='before lsted_scan_run'):
        h.frames(0, 1, [1] * 6, 0)
    h.run(np.pad(obj, ((0, 0), (4, 4), (4, 4))), 0, [0, 2])
    with pytest.raises(RuntimeError, match='outside the kept frames'):
        h.frames(1, 2, [1] * 6, 0)
    with pytest.raises(RuntimeError, match='ascending'):
        h.run(np.pad(obj, ((0, 0), (4, 4), (4, 4))), 0, [2, 0])
    h.close()


# --------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('name', SMALL + FULL)
def test_engine_on_gpu_against_reference_frames(name, golden):
    out, frames = run_case(engine().simulate_imaging, golden[1][name])
    check_against_golden(frames, name, golden)
    assert out['device_ms'] > 0


@pytest.mark.gpu
def test_helpers_on_gpu():
    check_helpers(engine())


@pytest.mark.gpu
def test_gpu_matches_oracle_on_a_tiled_object():
    """2x2 field of view of a 64^2 crop (line_sted_figure_3.py:46 tiles the object), rescan and
    descan line, 4 orientations: every orientation's final camera image / reconstruction."""
    obj = lines_object(64, tile=2)
    for typ in ('rescan_line', 'descan_line'):
        got = engine().simulate_imaging(obj, typ, 12, 2, 4, 1, 57, verbose=False)
        ref = scan_oracle.simulate_imaging(obj, typ, 12, 2, 4, 1, 57, keep_frames=False)
        assert len(got['orientations']) == 4
        for a, b in zip(got['orientations'], ref['orientations']):
            assert a['rot'] == b['rot'] and a['pulses_delivered'] == b['pulses_delivered']
            assert a['camera_exposures'] == b['camera_exposures']
            for k in ('reconstruction', 'cum_detector_sig'):
                assert np.abs(a[k] - b[k]).max() <= 1e-11 * np.abs(b[k]).max(), (typ, a['rot'], k)
        for k, v in ref['maxima'].items():
            assert abs(got['maxima'][k] - v) <= 1e-11 * abs(v), k


def test_rescan_line_with_long_columns_on_cpu_replay(emulated):
    """A frame tall enough (190 rows) for the blocked column prefilter of scale_y, excitation
    wide enough to reach the frame edges (no support limiting: reflect folds in both blur
    passes), two orientations: camera images and maxima against the oracle."""
    obj = lines_object(100)
    got = emulated.simulate_imaging(obj, 'rescan_line', 20, 1, 2, 1, 45, verbose=False)
    ref = scan_oracle.simulate_imaging(obj, 'rescan_line', 20, 1, 2, 1, 45, keep_frames=False)
    for a, b in zip(got['orientations'], ref['orientations']):
        assert a['rot'] == b['rot'] and a['camera_exposures'] == b['camera_exposures']
        for k in ('reconstruction', 'cum_detector_sig'):
            assert np.abs(a[k] - b[k]).max() <= 1e-11 * np.abs(b[k]).max(), (a['rot'], k)
    for k, v in ref['maxima'].items():
        assert abs(got['maxima'][k] - v) <= 1e-11 * abs(v), k


def compare_with_oracle(se, obj, typ, width, R, n_or, pad):
    frames = {}
    for name, sim in (('engine', se.simulate_imaging), ('oracle', oracle_sim)):
        got = []

        def record(filename, *a, got=got):
            got.append((os.path.basename(filename), [np.array(x) for x in a[:7]], a[7], a[8]))
        sim(obj, typ, width, R, n_or, 1, pad, comparison_name='case', generate_figure=record, verbose=False)
        frames[name] = got
    assert len(frames['engine']) == len(frames['oracle']) > 0
    for (fa, aa, pa, ca), (fb, ab, pb, cb) in zip(frames['engine'], frames['oracle']):
        assert fa.split('deg_')[1] == fb.split('deg_')[1] and pa == pb and ca == cb
        for x, y in zip(aa, ab):
            assert np.abs(x - y).max() <= TOL, fa


def test_point_scan_on_the_excitation_support_on_cpu_replay(emulated):
    """A descan-point scan whose excitation box and blur stay clear of the frame edges: both blur
    passes, the reductions and the glow maximum then work on that box only (the golden point case
    is too small for it).  Every drawn frame against the oracle."""
    obj = lines_object(24)
    h = emulated.ScanHandle('descan_point', obj.shape, 18, 8, 2)
    assert h.padded_shape == (60, 60) and len(h.positions) == 625
    h.close()
    compare_with_oracle(emulated, obj, 'descan_point', 8, 2, 1, 18)


@pytest.mark.gpu
def test_point_scan_on_the_excitation_support_on_gpu():
    compare_with_oracle(engine(), lines_object(24), 'descan_point', 8, 2, 1, 18)


@pytest.mark.parametrize('typ,n_or,pad', [('descan_point', 1, 9), ('nondescan_multipoint', 1, 9),
                                          ('descan_line', 2, 25), ('rescan_line', 2, 25)])
def test_rectangular_objects_on_cpu_replay(emulated, typ, n_or, pad):
    """Objects that are not square (rows != columns): every drawn frame against the oracle."""
    obj = lines_object(56)[:, 8:44, :].copy()        # 36 x 56
    compare_with_oracle(emulated, obj, typ, 9, 2, n_or, pad)
