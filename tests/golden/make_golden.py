#!/usr/bin/env python3
"""Generate the golden fixtures in this directory by running the UNMODIFIED
reference (`figure_generation/line_sted_tools.py`), read from
$LSTED_REFERENCE_DIR or baseline/_ref/ (tests/_reference_loader.py):
    python tests/golden/make_golden.py
Outputs (committed):
    psf_reports.npz      psf_report() dicts for four operating points
    fig2_2p0x_lr.npz     figure-2 '2p0x_lr' rescan line PSF, 4 orientations,
                         astronaut forward model + 8 RL iterations (seed 0)
    scalars.json         scalar goldens incl. tune_psf() results and the
                         numbers published in the reference's own documents
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from _reference_loader import load_reference, REFERENCE_DIR  # noqa: E402

ref = load_reference()
np_tif = sys.modules['np_tif']


def flatten_report(prefix, rep, store):
    scal = {}
    for k, v in rep.items():
        if k == 'psfs':
            for name, arr in v.items():
                store['%s/%s' % (prefix, name)] = arr
        else:
            scal[k] = float(v)
    return scal


def main():
    import scipy
    scalars = {'versions': {'numpy': np.__version__, 'scipy': scipy.__version__}}
    # ---- psf_report goldens ------------------------------------------------
    store = {}
    cases = {
        'point_1_9_8_1': ('point', 1, 9, 8, 1),
        'line_1_9_8_1': ('line', 1, 9, 8, 1),
        'line_0p25_3_12_2': ('line', 0.25, 3, 12, 2),
        'point_0p5_0_4_3': ('point', 0.5, 0, 4, 3),
    }
    scalars['psf_report'] = {}
    for name, args in cases.items():
        rep = ref.psf_report(*args, verbose=False)
        scalars['psf_report'][name] = {
            'args': list(args), **flatten_report(name, rep, store)}
    np.savez_compressed(os.path.join(HERE, 'psf_reports.npz'), **store)
    # ---- tune_psf goldens --------------------------------------------------
    scalars['tune_psf'] = {}
    for name, kw in {
        'point_R2_E4': dict(psf_type='point', scan_type='descanned',
                            desired_resolution_improvement=2.,
                            desired_emissions_per_molecule=4.,
                            max_excitation_brightness=0.25,
                            steps_per_improved_psf_width=4.),
        'line_rescanned_R2p2_E3': dict(psf_type='line', scan_type='rescanned',
                                       desired_resolution_improvement=2.2,
                                       desired_emissions_per_molecule=3.,
                                       max_excitation_brightness=0.25,
                                       steps_per_improved_psf_width=4.),
    }.items():
        res = ref.tune_psf(**kw)
        scalars['tune_psf'][name] = {
            'kwargs': kw,
            **{k: float(v) for k, v in res.items()
               if k not in ('psfs', 'psf_type', 'verbose', 'output_dir')}}
    # ---- figure-2 '2p0x_lr' forward model + RL -------------------------------
    p = dict(excitation_brightness=0.21672180512595912,
             depletion_brightness=11.766131198861775,
             steps_per_excitation_psf_width=25, pulses_per_position=5)
    fine = ref.psf_report('line', verbose=False, **p)
    base = fine['psfs']['rescan_sted']
    from scipy.ndimage import rotate as nd_rotate

    def rotate(x, degrees):  # line_sted_figure_2.py:264-272
        if degrees == 0:
            return x
        if degrees == 90:
            return np.rot90(np.squeeze(x)).reshape(x.shape)
        return np.clip(nd_rotate(x, angle=degrees, axes=(1, 2), reshape=False),
                       0, 1.1 * x.max())
    K = 4
    psfs = [1 / K * 3.0227 * rotate(base / base.sum(), a)
            for a in np.arange(0, 180, 180 / K)]
    obj = np_tif.tif_to_array(
        os.path.join(REFERENCE_DIR, 'test_object_astronaut.tif'))
    assert obj.dtype == np.uint8 and obj.shape == (1, 128, 128)
    d = ref.Deconvolver(psfs, output_prefix='/tmp/lsted_golden_', verbose=False)
    d.create_data_from_object(obj.astype(np.float64), total_brightness=5e10,
                              random_seed=0)
    out = {'object_u8': obj, 'base_psf': base,
           'psfs': np.concatenate(psfs, axis=0),
           'noiseless': np.concatenate(d.noiseless_measurement, axis=0),
           'noisy': np.concatenate(d.noisy_measurement, axis=0)}
    d.iterate()
    out['estimate_1'] = d.estimate.copy()
    out['H_t_normalization'] = d.H_t_normalization.copy()
    for _ in range(7):
        d.iterate()
    out['estimate_8'] = d.estimate.copy()
    np.savez_compressed(os.path.join(HERE, 'fig2_2p0x_lr.npz'), **out)
    scalars['fig2_2p0x_lr'] = {
        'psf_report_args': p, 'K': K, 'total_brightness': 5e10, 'seed': 0,
        'fine_line_report': {k: float(v) for k, v in fine.items() if k != 'psfs'},
        'noiseless0_sum': float(d.noiseless_measurement[0].sum()),
        'noisy0_sum': float(d.noisy_measurement[0].sum()),
        'estimate8_sum': float(d.estimate.sum()),
        'estimate8_max': float(d.estimate.max())}
    # ---- numbers published by the reference itself ---------------------------
    scalars['published'] = {
        'source': 'images/figure_1/point_1p00exc_9p00dep_008samps_001pulses.svg'
                  ':5928,6261,6455,6582 ; appendix.html:213-252',
        'point_1_9_8_1': {'excitation_dose': 72.52, 'depletion_dose': 2610.35,
                          'expected_emission': 3.39, 'resolution': 3.5},
        'fig2_point_rows': {  # R -> (exc dose, dep dose), emissions 4.00
            '1.5': [11.4, 500.3], '2.0': [18.8, 1696.8],
            '2.5': [30.3, 4159.5], '3.0': [46.7, 8601.8],
            '4.0': [90.7, 27044.0]},
    }
    with open(os.path.join(HERE, 'scalars.json'), 'w') as f:
        json.dump(scalars, f, indent=1, sort_keys=True)
    for fn in sorted(os.listdir(HERE)):
        print(fn, os.path.getsize(os.path.join(HERE, fn)))


if __name__ == '__main__':
    main()
