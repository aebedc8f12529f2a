"""Drop-in `line_sted_tools` backed by hand-written sm_100a CUDA kernels.

Same public names, argument order, defaults, return types and printed text as
`figure_generation/line_sted_tools.py` of AndrewGYork/rescan_line_sted
(cited below as ref:LINE), so the reference's figure scripts run on it
unchanged (numpy in, numpy out).  All array maths happens in liblsted.so
(see include/lsted.h) through ctypes.  A quiet `psf_report` (verbose=False, no
output_dir: what `tune_psf` and the figure sweeps call) is ONE kernel launch:
illumination, the Gaussian width fits of `get_width`, the integer rescan ratio,
the system PSFs and the doses all happen on the device; `tune_psf` keeps
scipy's Brent search on the host (every evaluation is that one launch), and
`tune_psf_batch` / `psf_report_batch` run many operating points per launch.
There is no CPU fallback for the array maths.

Backend switches (environment, read at call time; signatures unchanged):
  LSTED_PRECISION   fp32 (default) | fp64   storage/compute type of Deconvolver
  LSTED_DEVICE      CUDA device ordinal (default 0)
  LSTED_EXACT_CLIP  1 -> clip every H_t term before summing (ref:587) instead
                    of summing in the Fourier domain and clipping once
  LSTED_TILE_FFT    FFT length of overlap-save tiles (0/unset: tile only when the
                    padded object does not fit one shared-memory transform)
  LSTED_HOST_FIT    1 -> psf_report always fits widths with scipy's curve_fit on the
                    host (the reference's optimiser) instead of the device fit
"""
import os
import threading
import time

import numpy as np
from scipy.optimize import curve_fit, minimize_scalar

from . import _lib
from . import np_tif

__all__ = ['psf_report', 'generate_psfs', 'tune_psf', 'Deconvolver',
           'logarithmic_progress', 'get_width', 'psf_report_batch',
           'tune_psf_batch', 'get_width_batch']

_FWHM = 2 * np.sqrt(2 * np.log(2))


def _precision():
    p = os.environ.get('LSTED_PRECISION', 'fp32').lower()
    if p in ('fp32', '32', 'float32', 'single'):
        return 32
    if p in ('fp64', '64', 'float64', 'double'):
        return 64
    raise ValueError('LSTED_PRECISION must be fp32 or fp64, got %r' % p)


def _device():
    return int(os.environ.get('LSTED_DEVICE', '0'))


# ---------------------------------------------------------------------------
# PSF synthesis
# ---------------------------------------------------------------------------
def _gaussian_taps(sigma, truncate=4.0):
    """The FIR taps scipy.ndimage.gaussian_filter would use (order 0):
    radius int(truncate*sigma + 0.5), exp(-x^2/2s^2) normalised to sum 1."""
    sigma = float(sigma)
    radius = int(truncate * sigma + 0.5)
    x = np.arange(-radius, radius + 1)
    taps = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return np.ascontiguousarray(taps / taps.sum()), radius


def _grid(steps_per_excitation_psf_width):
    blur_sigma = steps_per_excitation_psf_width / _FWHM            # ref:91
    num_steps = 1 + 2 * int(np.round(5 * blur_sigma))               # ref:92
    return blur_sigma, num_steps


def _illumination(psf_type, n, blur_sigma, exc, dep):
    """Batched K1 kernel call -> dict of [B][n][n] arrays (ref:180-243)."""
    lib = _lib.get()
    taps, radius = _gaussian_taps(blur_sigma)
    exc = np.ascontiguousarray(np.atleast_1d(exc), dtype=np.float64)
    dep = np.ascontiguousarray(np.atleast_1d(dep), dtype=np.float64)
    B = exc.size
    names = ('excitation', 'depletion', 'excitation_fraction',
             'depletion_fraction', 'sted')
    out = {k: np.empty((B, n, n), dtype=np.float64) for k in names}
    p = _lib.c_double_p
    lib.call('lsted_psf_illumination', _device(),
             {'point': 0, 'line': 1}[psf_type], B, n, taps.ctypes.data_as(p),
             radius, exc.ctypes.data_as(p), dep.ctypes.data_as(p),
             *[out[k].ctypes.data_as(p) for k in names])
    return out


def _rescan(n, blur_sigma, sted_rows, ratios, want_wide=False):
    """Batched K2 kernel call (ref:258-310)."""
    lib = _lib.get()
    taps, radius = _gaussian_taps(blur_sigma)
    rows = np.ascontiguousarray(sted_rows, dtype=np.float64).reshape(-1, n)
    B = rows.shape[0]
    ratios = np.ascontiguousarray(ratios, dtype=np.int32).reshape(B)
    emission = np.empty((B, n, n))
    rescan = np.empty((B, n, n))
    descan = np.empty((B, n, n))
    wide = np.empty((1, n, int(ratios[0]) * n)) if want_wide else None
    p = _lib.c_double_p
    lib.call('lsted_psf_rescan', _device(), B, n, taps.ctypes.data_as(p),
             radius, rows.ctypes.data_as(p),
             ratios.ctypes.data_as(_lib.c_int_p), emission.ctypes.data_as(p),
             rescan.ctypes.data_as(p), descan.ctypes.data_as(p),
             wide.ctypes.data_as(p) if want_wide else None)
    return emission, rescan, descan, wide


def _rescan_ratio(sted_row, emission_sigma, verbose):
    line_sted_sigma, _ = get_width(sted_row)                       # ref:252
    ratio = (emission_sigma / line_sted_sigma) ** 2 + 1             # ref:254
    if verbose:
        print(" Ideal line rescan ratio: %0.5f" % (ratio))
    ratio = int(np.round(ratio))
    if verbose:
        print(" Neareset integer:", ratio)
    return ratio


def generate_psfs(
    shape,  # Desired pixel dimensions of the psfs
    excitation_brightness,  # Peak brightness in saturation units
    depletion_brightness,  # Peak brightness in saturation units
    blur_sigma,
    psf_type='point',
    output_dir=None,
    verbose=True,
    ):
    """Excitation / depletion / STED / system PSFs (ref:168-363) on the GPU.

    `shape` must be (1, n, n): the simulation is 2-D and `psf_report` only
    ever asks for square grids.
    """
    shape = tuple(int(s) for s in shape)
    if len(shape) != 3 or shape[0] != 1 or shape[1] != shape[2]:
        raise ValueError('generate_psfs: shape must be (1, n, n), got %r'
                         % (shape,))
    if psf_type not in ('point', 'line'):
        raise ValueError("psf_type must be 'point' or 'line'")
    n = shape[1]
    ill = _illumination(psf_type, n, blur_sigma, excitation_brightness,
                        depletion_brightness)
    psfs = {k: v for k, v in ill.items()}  # each (1, n, n)
    tifs = [('excitation', 'excitation_psf_%s.tif'),
            ('depletion', 'depletion_psf_%s.tif'),
            ('excitation_fraction', 'excitation_fraction_psf_%s.tif'),
            ('depletion_fraction', 'depletion_fraction_psf_%s.tif'),
            ('sted', 'sted_psf_%s.tif')]
    tifs = [(psfs[k], f % psf_type) for k, f in tifs]
    if psf_type == 'point':
        psfs['descan_sted'] = psfs['sted']  # Simple rename (ref:249)
    else:
        ratio = _rescan_ratio(psfs['sted'][0, n // 2, :], blur_sigma, verbose)
        if verbose:
            print(" Calculating rescan psf...", end='')
        emission, rescan, descan, wide = _rescan(
            n, blur_sigma, psfs['sted'][0, n // 2, :], [ratio],
            want_wide=output_dir is not None)
        if verbose:
            print(" ...done.")
        psfs['descan_sted'] = descan
        psfs['rescan_sted'] = rescan
        tifs += [(emission, 'emission_psf.tif'),
                 (wide, 'sted_psf_line_rescan_unscaled.tif'),
                 (rescan, 'sted_psf_line_rescan.tif'),
                 (descan, 'sted_psf_line_descan.tif')]
    if output_dir is not None:
        if not os.path.exists(output_dir):
            os.mkdir(output_dir)
        for array, filename in tifs:
            np_tif.array_to_tif(array, os.path.join(output_dir, filename))
    return psfs


def _report_from_psfs(psf_type, psfs, blur_sigma, num_steps,
                      pulses_per_position, verbose):
    """Widths, resolution factors, doses (ref:101-166)."""
    mid = num_steps // 2
    central_line_ex = psfs['excitation'][0, mid, :]
    central_line_st = psfs['sted'][0, mid, :]
    assert central_line_ex.max() == psfs['excitation'].max()
    assert central_line_st.max() == psfs['sted'].max()
    ex_sigma, _ = get_width(central_line_ex)
    sted_sigma, _ = get_width(central_line_st)
    res_descanned = blur_sigma / sted_sigma
    if verbose:
        print("PSF type:", psf_type)
        print("Excitation psf width: %0.3f" % (ex_sigma * _FWHM),
              "pixels FWHM")
        print("STED psf width: %0.3f" % (sted_sigma * _FWHM),
              "pixels FWHM")
        print("STED improvement in excitation PSF width: %0.3f" % (
            res_descanned))
    out = {}
    if psf_type == 'line':
        central_line_rescan = psfs['rescan_sted'][0, mid, :]
        assert central_line_rescan.max() == psfs['rescan_sted'].max()
        rescan_sigma, _ = get_width(central_line_rescan)
        res_rescanned = blur_sigma / rescan_sigma
        if verbose:
            print("Rescan STED psf width: %0.3f" % (rescan_sigma * _FWHM))
            print("Rescan STED improvement in PSF width: %0.3f" % (
                res_rescanned))
        out['resolution_improvement_rescanned'] = res_rescanned
        dose = lambda a: pulses_per_position * a[0, mid, :].sum()  # 1D scan
    else:
        dose = lambda a: pulses_per_position * a.sum()             # 2D scan
    out['resolution_improvement_descanned'] = res_descanned
    out['excitation_dose'] = dose(psfs['excitation'])
    out['depletion_dose'] = dose(psfs['depletion'])
    out['expected_emission'] = dose(psfs['sted'])
    out['pulses_per_position'] = pulses_per_position
    out['psfs'] = psfs
    if verbose:
        print("Excitation dose: %0.3f" % (out['excitation_dose']),
              "half-saturations")
        print("Depletion dose: %0.3f" % (out['depletion_dose']),
              "half-saturations")
        print("Expected emissions per molecule: %0.4f\n" % (
            out['expected_emission']))
    return out


# scalar slots of lsted_psf_report_batch (include/lsted.h)
(_PR_EX_SIGMA, _PR_STED_SIGMA, _PR_RESCAN_SIGMA, _PR_RATIO_REAL, _PR_RATIO,
 _PR_EXC_DOSE, _PR_DEP_DOSE, _PR_EMISSION, _PR_FIT_ITERS, _PR_FIT_STATUS,
 _PR_EX_MAX_OK, _PR_STED_MAX_OK, _PR_RESCAN_MAX_OK) = range(13)
_PR_SCALARS = 16
_PSF_PLANES = ('excitation', 'depletion', 'excitation_fraction',
               'depletion_fraction', 'sted', 'rescan_sted', 'descan_sted')
# The device fit restates scipy's optimiser (MINPACK lmdif) step for step; on the GPU only
# exp() may differ in the last place.  A fitted rescan ratio this close (relative) to a
# rounding boundary k + 1/2 is still left to scipy itself: the integer decides array shapes.
_RATIO_TIE_BAND = 1e-6
# A profile narrower than this (pixels) is essentially one sample: its fitted "width" is
# whatever the optimiser's rounding noise makes it (scipy's own answer moves by tens of per
# cent with a last-place change of the data -- 0.28 or 0.13 px for the same profile), so
# the reference's optimiser itself decides.  tune_psf samples >= 3 steps per width: never.
_ILL_POSED_SIGMA = 0.35
_taps_cache = {}


def _host_fit_forced():
    return os.environ.get('LSTED_HOST_FIT', '0') not in ('', '0')


def _device_reports(psf_type, exc, dep, steps, pulses, want_psfs):
    """The fused K1+K2+fit kernel for B operating points (each with its own
    sampling): list of `psf_report` dicts, or None where the point has to be
    redone with the host fit (rescan ratio within 1e-6 of a rounding boundary,
    or a fit that did not converge)."""
    lib = _lib.get()
    B = len(exc)
    grids = [_grid(st) for st in steps]
    taps = []
    for sigma, _ in grids:
        if sigma not in _taps_cache:
            if len(_taps_cache) > 4096:
                _taps_cache.clear()
            _taps_cache[sigma] = _gaussian_taps(sigma)
        taps.append(_taps_cache[sigma])
    tap_stride = max(len(t) for t, _ in taps)
    tap_block = np.zeros((B, tap_stride))
    for b, (t, _) in enumerate(taps):
        tap_block[b, :len(t)] = t
    n = np.array([g[1] for g in grids], dtype=np.int32)
    radius = np.array([r for _, r in taps], dtype=np.int32)
    sigma = np.array([g[0] for g in grids], dtype=np.float64)
    exc = np.ascontiguousarray(exc, dtype=np.float64)
    dep = np.ascontiguousarray(dep, dtype=np.float64)
    nmax = int(n.max())
    scalars = np.empty((B, _PR_SCALARS))
    planes = np.empty((B, 7, nmax * nmax)) if want_psfs else None
    p = _lib.c_double_p
    lib.call('lsted_psf_report_batch', _device(),
             {'point': 0, 'line': 1}[psf_type], B,
             n.ctypes.data_as(_lib.c_int_p), radius.ctypes.data_as(_lib.c_int_p),
             tap_block.ctypes.data_as(p), tap_stride, sigma.ctypes.data_as(p),
             exc.ctypes.data_as(p), dep.ctypes.data_as(p),
             scalars.ctypes.data_as(p),
             planes.ctypes.data_as(p) if want_psfs else None)
    reports = []
    for b in range(B):
        sc = scalars[b]
        nb = int(n[b])
        if sc[_PR_FIT_STATUS] != 0:
            reports.append(None)
            continue
        widths = [sc[_PR_EX_SIGMA], sc[_PR_STED_SIGMA]] + (
            [sc[_PR_RESCAN_SIGMA]] if psf_type == 'line' else [])
        if min(abs(w) for w in widths) < _ILL_POSED_SIGMA:
            reports.append(None)
            continue
        if psf_type == 'line':
            frac = sc[_PR_RATIO_REAL] - np.floor(sc[_PR_RATIO_REAL])
            if abs(frac - 0.5) < _RATIO_TIE_BAND * max(1.0, sc[_PR_RATIO_REAL]):
                reports.append(None)
                continue
        # the reference's exact-equality asserts (ref:105-106, :120)
        assert sc[_PR_EX_MAX_OK] == 1 and sc[_PR_STED_MAX_OK] == 1
        assert sc[_PR_RESCAN_MAX_OK] == 1
        out = {}
        if psf_type == 'line':
            out['resolution_improvement_rescanned'] = (
                sigma[b] / sc[_PR_RESCAN_SIGMA])
        out['resolution_improvement_descanned'] = sigma[b] / sc[_PR_STED_SIGMA]
        out['excitation_dose'] = pulses[b] * sc[_PR_EXC_DOSE]
        out['depletion_dose'] = pulses[b] * sc[_PR_DEP_DOSE]
        out['expected_emission'] = pulses[b] * sc[_PR_EMISSION]
        out['pulses_per_position'] = pulses[b]
        if want_psfs:
            names = _PSF_PLANES if psf_type == 'line' else _PSF_PLANES[:5]
            psfs = {k: planes[b, i, :nb * nb].reshape(1, nb, nb).copy()
                    for i, k in enumerate(names)}
            if psf_type == 'point':
                psfs['descan_sted'] = psfs['sted']  # Simple rename (ref:249)
            out['psfs'] = psfs
        reports.append(out)
    return reports


def _host_fit_report(psf_type, excitation_brightness, depletion_brightness,
                     steps_per_excitation_psf_width, pulses_per_position,
                     verbose, output_dir):
    """psf_report with the widths fitted by scipy on the host (prints and TIFF
    side outputs included): three launches and 3-4 `curve_fit`s."""
    blur_sigma, num_steps = _grid(steps_per_excitation_psf_width)
    psfs = generate_psfs(
        shape=(1, num_steps, num_steps),
        excitation_brightness=excitation_brightness,
        depletion_brightness=depletion_brightness,
        blur_sigma=blur_sigma,
        psf_type=psf_type,
        verbose=verbose,
        output_dir=output_dir)
    return _report_from_psfs(psf_type, psfs, blur_sigma, num_steps,
                             pulses_per_position, verbose)


_evaluator = threading.local()   # set by tune_psf_batch: evaluations go to a shared batch


def _quiet_report(psf_type, excitation_brightness, depletion_brightness,
                  steps_per_excitation_psf_width, pulses_per_position,
                  want_psfs=True):
    """One quiet operating point: the fused device path (through the batch
    rendezvous when tune_psf_batch runs this thread), host fit as tie-breaker."""
    if _host_fit_forced():
        return _host_fit_report(psf_type, excitation_brightness,
                                depletion_brightness,
                                steps_per_excitation_psf_width,
                                pulses_per_position, False, None)
    point = (psf_type, float(excitation_brightness), float(depletion_brightness),
             steps_per_excitation_psf_width, pulses_per_position, want_psfs)
    batch = getattr(_evaluator, 'rendezvous', None)
    if batch is not None:
        rep = batch.submit(point)
    else:
        rep = _device_reports(psf_type, [point[1]], [point[2]], [point[3]],
                              [point[4]], want_psfs)[0]
    if rep is None:
        rep = _host_fit_report(psf_type, excitation_brightness,
                               depletion_brightness,
                               steps_per_excitation_psf_width,
                               pulses_per_position, False, None)
    return rep


def psf_report(
    psf_type,  # Point or line
    excitation_brightness,  # Peak brightness in saturation units
    depletion_brightness,  # Peak brightness in saturation units
    steps_per_excitation_psf_width,  # Too small? Bad res. Too big? Excess dose.
    pulses_per_position,  # Think of this as "dwell time"
    verbose=True,
    output_dir=None,
    ):
    """One operating point: PSFs, resolution improvement, dose (ref:75-166)."""
    if psf_type not in ('point', 'line'):
        raise ValueError("psf_type must be 'point' or 'line'")
    if verbose or output_dir is not None:
        # the progress prints of generate_psfs sit between its stages
        return _host_fit_report(psf_type, excitation_brightness,
                                depletion_brightness,
                                steps_per_excitation_psf_width,
                                pulses_per_position, verbose, output_dir)
    return _quiet_report(psf_type, excitation_brightness, depletion_brightness,
                         steps_per_excitation_psf_width, pulses_per_position)


def psf_report_batch(psf_type, excitation_brightness, depletion_brightness,
                     steps_per_excitation_psf_width, pulses_per_position,
                     psfs=True):
    """Extension (not in the reference): many operating points in ONE kernel
    launch (one CTA each; samplings may differ from point to point).  Returns
    a list of `psf_report` dicts equal to calling `psf_report(...,
    verbose=False)` per point; `psfs=False` leaves the arrays on the device
    (scalars only)."""
    exc, dep, steps, pulses = np.broadcast_arrays(
        np.atleast_1d(np.asarray(excitation_brightness, dtype=np.float64)),
        np.atleast_1d(np.asarray(depletion_brightness, dtype=np.float64)),
        np.atleast_1d(steps_per_excitation_psf_width),
        np.atleast_1d(pulses_per_position))
    exc, dep, steps, pulses = (a.ravel() for a in (exc, dep, steps, pulses))
    if _host_fit_forced():
        reports = [None] * exc.size
    else:
        reports = _device_reports(psf_type, exc, dep, steps, pulses, psfs)
    for b, rep in enumerate(reports):
        if rep is None:
            reports[b] = _host_fit_report(psf_type, exc[b], dep[b], steps[b],
                                          pulses[b], False, None)
    return reports


def tune_psf(
    psf_type,  # 'point' or 'line'
    scan_type,  # 'descanned' or 'rescanned'
    desired_resolution_improvement,
    desired_emissions_per_molecule,
    max_excitation_brightness=0.5,  # Saturation units
    steps_per_improved_psf_width=3,
    relative_error=1e-6,
    verbose_results=False,
    verbose_iterations=False,
    ):
    """Solve for (depletion, pulses, excitation) that reach a target
    resolution improvement and emission level (ref:365-476): alternate two
    1-D Brent searches, every evaluation being one GPU `psf_report`."""
    assert (psf_type, scan_type) in (('point', 'descanned'),
                                     ('line', 'descanned'),
                                     ('line', 'rescanned'))
    for v in (desired_resolution_improvement, desired_emissions_per_molecule,
              max_excitation_brightness, steps_per_improved_psf_width,
              relative_error):
        assert float(v) == v
    res_key = 'resolution_improvement_' + scan_type
    args = {  # The inputs to psf_report()
        'psf_type': psf_type,
        'excitation_brightness': max_excitation_brightness,
        'depletion_brightness': 1,
        'steps_per_excitation_psf_width': (steps_per_improved_psf_width *
                                           desired_resolution_improvement),
        'pulses_per_position': 1,
        'verbose': False,
        'output_dir': None}

    def report(want_psfs):
        # (args carries verbose=False, output_dir=None: the quiet, single-launch path;
        # the searches only need scalars, so the PSF arrays stay on the device)
        return _quiet_report(args['psf_type'], args['excitation_brightness'],
                             args['depletion_brightness'],
                             args['steps_per_excitation_psf_width'],
                             args['pulses_per_position'], want_psfs)

    def resolution_error(depletion_brightness):
        args['depletion_brightness'] = abs(depletion_brightness)
        return (report(False)[res_key] -
                desired_resolution_improvement) ** 2

    def emission_error(excitation_brightness):
        args['excitation_brightness'] = abs(excitation_brightness)
        return (report(False)['expected_emission'] -
                desired_emissions_per_molecule) ** 2

    num_iterations = 0
    while True:
        num_iterations += 1
        if num_iterations >= 10:
            print("Max. iterations exceeded; giving up")
            break
        # Depletion brightness sets the resolution:
        args['depletion_brightness'] = abs(minimize_scalar(resolution_error).x)
        if verbose_iterations:
            print("Depletion brightness:", args['depletion_brightness'])
        # Pulse count from the emission of a single pulse pair:
        args['excitation_brightness'] = max_excitation_brightness
        args['pulses_per_position'] = 1
        results = report(False)
        args['pulses_per_position'] = np.ceil(
            desired_emissions_per_molecule / results['expected_emission'])
        if verbose_iterations:
            print(args['pulses_per_position'], "pulses.")
        # Excitation brightness trims the emission:
        args['excitation_brightness'] = abs(minimize_scalar(emission_error).x)
        if verbose_iterations:
            print("Excitation brightness:", args['excitation_brightness'])
        results = report(True)
        # Excitation saturation nudges the resolution; go round again if the
        # resolution drifted (one-sided test, like ref:461).
        relative_resolution_error = (
            (results[res_key] - desired_resolution_improvement) /
            desired_resolution_improvement)
        if relative_resolution_error < relative_error:
            break
    if verbose_results:  # same text as ref:463-474
        print("PSF tuning complete, after", num_iterations, "iterations.")
        for title, table in ((" Inputs:", args), (" Outputs:", results)):
            print(title)
            for k in sorted(table):
                shown = sorted(table[k].keys()) if k == 'psfs' else table[k]
                print('  ', k, ': ', shown, sep='')
        print()
    results.update(args)  # Combine the two dictionaries
    return results


class _Rendezvous:
    """Meeting point of the worker threads of `tune_psf_batch`: every thread
    hands in the operating point its search wants next and sleeps; when all
    live threads have one pending, the last arrival runs them as ONE batched
    kernel launch per PSF type and wakes the others."""

    def __init__(self, workers):
        self.cond = threading.Condition()
        self.live = workers
        self.pending = []          # [point, result, done, error]

    def submit(self, point):
        slot = [point, None, False, None]
        with self.cond:
            self.pending.append(slot)
            if len(self.pending) >= self.live:
                self._flush()
            while not slot[2]:
                self.cond.wait()
        if slot[3] is not None:
            raise slot[3]
        return slot[1]

    def retire(self):
        with self.cond:
            self.live -= 1
            if self.pending and len(self.pending) >= self.live:
                self._flush()

    def _flush(self):   # (lock held)
        slots, self.pending = self.pending, []
        groups = {}
        for sl in slots:
            groups.setdefault((sl[0][0], sl[0][5]), []).append(sl)
        for (psf_type, want_psfs), group in groups.items():
            try:
                reps = _device_reports(psf_type, [g[0][1] for g in group],
                                       [g[0][2] for g in group],
                                       [g[0][3] for g in group],
                                       [g[0][4] for g in group], want_psfs)
                for g, rep in zip(group, reps):
                    g[1] = rep
            except Exception as e:   # every waiter of the group sees it
                for g in group:
                    g[3] = e
            for g in group:
                g[2] = True
        self.cond.notify_all()


def tune_psf_batch(targets, max_concurrent=256):
    """Extension (not in the reference): `[tune_psf(**t) for t in targets]`
    with the operating points of all searches evaluated together -- each
    target keeps its own (strictly sequential) Brent searches, run by scipy in
    a thread of its own, and every round of evaluations is one batched kernel
    launch (one CTA per target) instead of one launch per evaluation.  Results
    are identical to calling `tune_psf` per target.

    targets: iterable of dicts of `tune_psf` keyword arguments."""
    targets = [dict(t) for t in targets]
    results = [None] * len(targets)
    errors = [None] * len(targets)
    for first in range(0, len(targets), max_concurrent):
        chunk = range(first, min(first + max_concurrent, len(targets)))
        meet = _Rendezvous(len(chunk))

        def work(i):
            _evaluator.rendezvous = meet
            try:
                results[i] = tune_psf(**targets[i])
            except BaseException as e:
                errors[i] = e
            finally:
                _evaluator.rendezvous = None
                meet.retire()

        threads = [threading.Thread(target=work, args=(i,)) for i in chunk]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
    for e in errors:
        if e is not None:
            raise e
    return results


# ---------------------------------------------------------------------------
# Forward model + multi-view Richardson-Lucy
# ---------------------------------------------------------------------------
def _stack_psfs(psfs):
    """List of (1, ny, nx) arrays -> one [K][ny][nx] block.  PSFs of unequal
    size are zero-padded so that the 'same' crop offset (n-1)//2 of each
    moves with its centre (the convolution result is unchanged)."""
    arrs = []
    for p in psfs:
        p = np.asarray(p, dtype=np.float64)
        if p.ndim == 2:
            p = p[None]
        if p.ndim != 3 or p.shape[0] != 1:
            raise ValueError('each PSF must have shape (1, ny, nx); got %r'
                             % (p.shape,))
        arrs.append(p[0])
    ny = max(a.shape[0] for a in arrs)
    nx = max(a.shape[1] for a in arrs)
    out = np.zeros((len(arrs), ny, nx))
    for k, a in enumerate(arrs):
        before = []
        for n_old, n_new in ((a.shape[0], ny), (a.shape[1], nx)):
            before.append((n_new - 1) // 2 - (n_old - 1) // 2)
        out[k, before[0]:before[0] + a.shape[0],
            before[1]:before[1] + a.shape[1]] = a
    return out


class Deconvolver:
    """GPU-resident counterpart of the reference `Deconvolver` (ref:478-594).

    `true_object`, `noiseless_measurement`, `noisy_measurement`, `estimate`
    and `H_t_normalization` live in HBM; reading the attribute copies to a
    fresh numpy array, assigning `noisy_measurement` / `estimate` uploads
    (that is the injection point for a given noise field).  Arrays handed
    out are copies: mutate-in-place does not write through, assign instead.

    CUDA tensors (float32 or float64, C-contiguous, on the handle's device)
    take a path without host copies, ordered on the current torch stream:
    `create_data_from_object`, `H` and `H_t` accept them and return tensors,
    the `noisy_measurement` / `estimate` setters accept them, and
    `tensor(name)` reads an attribute as tensors.
    """

    def __init__(self, psfs, output_prefix=None, verbose=True):
        self.psfs = list(psfs)
        if output_prefix is None:
            output_prefix = os.getcwd()
        if not os.path.exists(os.path.dirname(output_prefix)):
            os.mkdir(os.path.dirname(output_prefix))
        self.output_prefix = output_prefix
        self.verbose = verbose
        self.num_iterations = 0
        self.saved_iterations = []
        self.estimate_history = []
        self._handle = None
        self._shape = None
        self._psf_key = None
        self._have = set()  # which device arrays hold data
        self._data_version = 0  # bumped whenever true_object changes

    # -- device plumbing ----------------------------------------------------
    def _engine(self, shape):
        """Handle for images of `shape` = (1, Ny, Nx); (re)built on demand."""
        shape = tuple(int(s) for s in shape)
        if len(shape) != 3 or shape[0] != 1:
            raise ValueError('images must have shape (1, Ny, Nx); got %r'
                             % (shape,))
        # The reference reads self.psfs on every H / H_t call (ref:573, :585): a replaced
        # list or replaced arrays rebuild the OTFs (in-place edits of an array's contents
        # are not seen -- assign a new array instead).
        psf_key = tuple(id(p) for p in self.psfs)
        if (self._handle is None or self._shape != shape
                or self._psf_key != psf_key):
            keep = {}
            if self._handle is not None:
                if self._shape == shape:   # same images, new PSFs: the state carries over
                    K_new = len(self.psfs)
                    # (H_t_normalization included: the reference caches it once, ref:590-592)
                    for which in sorted(self._have):
                        per_psf = which in (_lib.NOISELESS, _lib.NOISY)
                        if per_psf and K_new != self._handle.K:
                            continue
                        keep[which] = [self._handle.get(which, k) for k in
                                       range(self._handle.K if per_psf else 1)]
                self._handle.close()
            self._handle = _lib.DeconvHandle(
                _lib.get(), _stack_psfs(self.psfs), shape[1:],
                precision=_precision(), device=_device(),
                tile_fft_len=int(os.environ.get('LSTED_TILE_FFT', '0') or 0))
            if os.environ.get('LSTED_EXACT_CLIP', '0') not in ('', '0'):
                self._handle.set_option('exact_clip', 1)
            self._shape = shape
            self._psf_key = psf_key
            self._have = set()
            for which, arrays in keep.items():
                for k, a in enumerate(arrays):
                    self._handle.set(which, k, a)
                self._have.add(which)
        return self._handle

    def _check_tensor(self, t, what):
        """A (1, Ny, Nx) CUDA tensor on the handle's device (checked before any
        handle is built or any call crosses into the library)."""
        device = self._handle.device if self._handle is not None else _device()
        return _lib.check_tensor(t, (1, None, None), device, what)

    def _need(self, what, name):
        if self._handle is None or what not in self._have:
            raise AttributeError("'Deconvolver' object has no attribute '%s'"
                                 % name)
        return self._engine(self._shape)   # (notices replaced PSFs)

    @property
    def true_object(self):
        return self._need(_lib.TRUE_OBJECT, 'true_object').get(_lib.TRUE_OBJECT)

    @property
    def noiseless_measurement(self):
        h = self._need(_lib.NOISELESS, 'noiseless_measurement')
        return [h.get(_lib.NOISELESS, k) for k in range(h.K)]

    @property
    def noisy_measurement(self):
        h = self._need(_lib.NOISY, 'noisy_measurement')
        return [h.get(_lib.NOISY, k) for k in range(h.K)]

    @noisy_measurement.setter
    def noisy_measurement(self, value):
        value = list(value)
        if value and _lib.is_tensor(value[0]):
            if len(value) != len(self.psfs):
                raise ValueError('need one measurement per PSF')
            for v in value:
                self._check_tensor(v, 'each measurement')
            h = self._engine(value[0].shape)
            for k, v in enumerate(value):
                h.set_tensor(_lib.NOISY, k, v)
            self._have.add(_lib.NOISY)
            return
        value = [np.asarray(v, dtype=np.float64) for v in value]
        if len(value) != len(self.psfs):
            raise ValueError('need one measurement per PSF')
        h = self._engine(value[0].shape if value[0].ndim == 3
                         else (1,) + value[0].shape)
        for k, v in enumerate(value):
            h.set(_lib.NOISY, k, v)
        self._have.add(_lib.NOISY)

    @property
    def estimate(self):
        return self._need(_lib.ESTIMATE, 'estimate').get(_lib.ESTIMATE)

    @estimate.setter
    def estimate(self, value):
        if _lib.is_tensor(value):
            self._check_tensor(value, 'estimate')
            self._engine(value.shape).set_tensor(_lib.ESTIMATE, 0, value)
        else:
            value = np.asarray(value, dtype=np.float64)
            h = self._engine(value.shape)
            h.set(_lib.ESTIMATE, 0, value)
        self._have.add(_lib.ESTIMATE)

    @property
    def H_t_normalization(self):
        return self._need(_lib.NORMALIZATION,
                          'H_t_normalization').get(_lib.NORMALIZATION)

    _ATTRIBUTES = {'true_object': _lib.TRUE_OBJECT,
                   'noiseless_measurement': _lib.NOISELESS,
                   'noisy_measurement': _lib.NOISY,
                   'estimate': _lib.ESTIMATE,
                   'H_t_normalization': _lib.NORMALIZATION}

    def tensor(self, name, dtype=None):
        """Extension: attribute `name` as CUDA tensors of `dtype` (torch.float64 by
        default) on the handle's device, without a host copy -- a (1, Ny, Nx)
        tensor, or for the per-PSF measurements a list of (1, Ny, Nx) views of one
        (K, Ny, Nx) tensor.  Ordered on the current torch stream."""
        import torch
        if name not in self._ATTRIBUTES:
            raise ValueError('tensor(): name must be one of %s, got %r'
                             % (', '.join(sorted(self._ATTRIBUTES)), name))
        dtype = torch.float64 if dtype is None else dtype
        if dtype not in (torch.float32, torch.float64):
            raise TypeError('tensor(): dtype must be torch.float32 or torch.float64')
        which = self._ATTRIBUTES[name]
        h = self._need(which, name)
        if which not in (_lib.NOISELESS, _lib.NOISY):
            return h.get_tensor(which, 0, dtype)
        out = torch.empty((h.K, h.Ny, h.Nx), dtype=dtype,
                          device=torch.device('cuda', h.device))
        for k in range(h.K):
            h.get_tensor(which, k, out=out[k:k + 1])
        return [out[k:k + 1] for k in range(h.K)]

    # -- the reference's methods ---------------------------------------------
    def create_data_from_object(
        self,
        obj,
        total_brightness=None,
        random_seed=None
        ):
        """Forward model + shot noise (ref:496-512).  The Poisson field comes
        from the in-kernel Philox generator: `random_seed` selects its
        stream; without a seed one is drawn from numpy's global generator
        (so `np.random.seed` upstream still makes a run repeatable).
        `obj` may be a float32 / float64 CUDA tensor of shape (1, Ny, Nx)."""
        tensor = _lib.is_tensor(obj)
        if tensor:
            self._check_tensor(obj, 'obj')
        assert len(obj.shape) == 3
        assert tensor or obj.dtype == np.float64
        h = self._engine(obj.shape)
        if random_seed is None:
            random_seed = int(np.random.randint(0, 2 ** 31 - 1)) * 2 ** 31 + \
                int(np.random.randint(0, 2 ** 31 - 1))
        # like the reference, new data leave `estimate` and `num_iterations` alone
        if tensor:
            h.upload_object_tensor(obj)
            h.simulate(total_brightness, int(random_seed) % 2 ** 64, reset_estimate=False)
        else:
            h.create_data(obj, total_brightness, int(random_seed) % 2 ** 64,
                          reset_estimate=False)
        self._data_version += 1
        self._have |= {_lib.TRUE_OBJECT, _lib.NOISELESS, _lib.NOISY}
        return None

    def load_data_from_tif(self, filename):
        """ref:514-518 (the reference's shape assertion `shape == 3` can
        never hold; this version checks the intent, a 3-D stack)."""
        data = np_tif.tif_to_array(filename).astype(np.float64) + 1e-9
        assert len(data.shape) == 3
        assert data.min() >= 0
        self.noisy_measurement = [data[k:k + 1] for k in range(data.shape[0])]
        return None

    def iterate(self):
        """One multi-view Richardson-Lucy update on the GPU (ref:520-531)."""
        h = self._need(_lib.NOISY, 'noisy_measurement')
        if self.num_iterations == 0:   # ref:521-522: the first call always starts from ones
            h.set_option('reset_estimate', 1)
        h.iterate(1)
        self.num_iterations += 1
        self._have |= {_lib.ESTIMATE, _lib.NORMALIZATION}
        return None

    def iterate_many(self, n):
        """Extension: n RL updates without returning to Python in between."""
        h = self._need(_lib.NOISY, 'noisy_measurement')
        if self.num_iterations == 0 and int(n) > 0:
            h.set_option('reset_estimate', 1)
        h.iterate(int(n))
        self.num_iterations += int(n)
        self._have |= {_lib.ESTIMATE, _lib.NORMALIZATION}

    def record_iteration(self, save_tifs=True):
        """ref:533-548: keep a copy of the estimate; rewrite the history
        TIFFs (estimate and log-magnitude spectrum of its error)."""
        self.saved_iterations.append(self.num_iterations)
        self.estimate_history.append(self.estimate)
        if save_tifs:
            eh = np.squeeze(np.concatenate(self.estimate_history, axis=0))
            np_tif.array_to_tif(eh, self.output_prefix + 'estimate_history.tif')
            # The reference re-transforms the whole history on every call (ref:539-548);
            # the spectra of the estimates already saved cannot change, so only the new
            # ones are computed -- same file, linear instead of quadratic work.
            cache = self.__dict__.setdefault('_ft_error_history', [])
            if cache and cache[0][0] != self._data_version:
                del cache[:]                       # new object: start over
            if len(cache) < len(self.estimate_history):
                # on the device (un-padded 2-D transform + log-magnitude + fftshift in the
                # column kernel's epilogue; sides without a Stockham plan and tiled objects take
                # the direct transform of ew_bodies.cuh) -- there is no host transform
                h = self._need(_lib.TRUE_OBJECT, 'true_object')
                first_new = len(cache)
                for i, est in enumerate(self.estimate_history[first_new:], first_new):
                    newest = i == len(self.estimate_history) - 1   # = the estimate in HBM
                    spectrum = h.ft_error(None if newest else est)
                    if spectrum is None:       # a rank of a sharded object: the gathered estimate
                        spectrum = h.ft_error(est)
                    if spectrum is None:
                        raise RuntimeError('lsted_deconv_ft_error: no device transform ran')
                    cache.append((self._data_version, spectrum))
            spectrum = np.concatenate([c[1] for c in cache], axis=0)
            np_tif.array_to_tif(
                spectrum, self.output_prefix + 'estimate_FT_error_history.tif')
        return None

    def record_data(self):
        """ref:550-565: dump psfs / object / measurements as TIFFs (whatever of
        them exists so far)."""
        def stack(arrays):
            return np.squeeze(np.concatenate(arrays, axis=0))
        outputs = (('psfs', 'psfs.tif', stack),
                   ('true_object', 'object.tif', lambda a: a),
                   ('noiseless_measurement', 'noiseless_measurement.tif', stack),
                   ('noisy_measurement', 'noisy_measurement.tif', stack))
        for attribute, filename, prepare in outputs:
            if hasattr(self, attribute):
                np_tif.array_to_tif(prepare(getattr(self, attribute)),
                                    self.output_prefix + filename)
        return None

    def H(self, x):
        """Expected noiseless measurement operator (ref:567-577): one
        clipped linear 'same' convolution per PSF, as a list.  A CUDA tensor
        gives views of one (K, Ny, Nx) tensor of its dtype."""
        if _lib.is_tensor(x):
            self._check_tensor(x, 'x')
            out = self._engine(x.shape).H_tensor(x)
            return [out[k:k + 1] for k in range(out.shape[0])]
        x = np.asarray(x, dtype=np.float64)
        h = self._engine(x.shape)
        out = h.H(x)
        return [out[k:k + 1] for k in range(h.K)]

    def H_t(self, y, normalize=True):
        """Transpose operator (ref:579-594), by default normalised so that
        H_t(ones) == ones.  A list of CUDA tensors gives a tensor."""
        y = list(y)
        if y and _lib.is_tensor(y[0]):
            for v in y:
                self._check_tensor(v, 'each image of y')
            if len({(v.shape, v.dtype) for v in y}) != 1:
                raise ValueError('the images of y must share one shape and dtype')
            h = self._engine(y[0].shape)
            if len(y) != h.K:
                raise ValueError('need one image per PSF (%d), got %d' % (h.K, len(y)))
            import torch
            out = h.Ht_tensor(torch.cat(y, dim=0), normalize)
        else:
            y = [np.asarray(v, dtype=np.float64) for v in y]
            h = self._engine(y[0].shape)
            out = h.Ht(np.concatenate(y, axis=0), normalize)
        if normalize:
            self._have.add(_lib.NORMALIZATION)
        return out


def logarithmic_progress(iterable, verbose=True):
    """Yield (item, flag); flag is True on indices 1, 2, 4, ... and on the
    last one.  Prints a coarse progress bar once the loop has run for more
    than 1.5 s (ref:596-651)."""
    total = len(iterable)
    if total == 0:
        return iterable
    save, i = [], 0
    while 2 ** i + 1 < total:
        save.append(2 ** i)
        i += 1
    save.append(total - 1)
    bar = ("Progress:\n|0%" + " " * 13 + "|" + " " * 15 + "|50%" + " " * 12 +
           "|" + " " * 15 + "|100%")
    bar_printed, stars_printed = False, 0
    start_time = time.perf_counter()
    for i, x in enumerate(iterable):
        yield (x, i in save)
        if not verbose:
            continue
        elapsed = time.perf_counter() - start_time
        if elapsed > 1.5:
            if i in save:
                rate = i / elapsed
                remaining = (total - i) / rate
                print("Iteration ", i, "/", total - 1,
                      " %0.1fs elapsed, " % (elapsed),
                      "~%0.1fs remaining, " % (remaining),
                      "%0.1f iter/s\n" % (rate),
                      sep='', end='')
                bar_printed, stars_printed = False, 0
            if not bar_printed:
                print(bar)
                bar_printed = True
            while stars_printed / 65 < i / total:
                print("*", end='')
                stars_printed += 1
            if (i + 1) in save:
                print()


def get_width_batch(rows):
    """Extension (not in the reference): `get_width` of many profiles of one length in one
    launch -- the in-kernel restatement of scipy's optimiser (MINPACK lmdif from
    p0 = [1, len/2, 1] at curve_fit's default tolerances).  Returns the widths [B] and the
    fitted (A, mu, sigma) [B][3]; raises like curve_fit where MINPACK does not converge."""
    rows = np.ascontiguousarray(rows, dtype=np.float64)
    if rows.ndim == 1:
        rows = rows[None]
    out = np.empty((rows.shape[0], 5))
    p = _lib.c_double_p
    _lib.get().call('lsted_gauss_fit', _device(), rows.shape[0], rows.shape[1],
                    rows.ctypes.data_as(p), out.ctypes.data_as(p))
    bad = ~((out[:, 4] >= 1) & (out[:, 4] <= 4))
    if bad.any():
        raise RuntimeError('Optimal parameters not found: MINPACK info %d for profile %d'
                           % (int(out[bad, 4][0]), int(np.flatnonzero(bad)[0])))
    return out[:, 2].copy(), out[:, :3].copy()


def get_width(x):
    """Width of a 1-D profile from a Gaussian fit (ref:653-668):
    Levenberg-Marquardt on A*exp(-(x-mu)^2/(2 sigma^2)), p0=[1, len/2, 1].
    A 3-parameter scalar fit on <=135 samples: host side, like the
    reference."""
    def gauss(x, *p):
        A, mu, sigma = p
        return A * np.exp(-(x - mu) ** 2 / (2. * sigma ** 2))
    coords = range(len(x))
    coeff, _ = curve_fit(gauss, coords, x, p0=[1., len(x) / 2., 1.])
    return coeff[2], gauss(coords, *coeff)
