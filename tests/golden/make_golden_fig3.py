#!/usr/bin/env python3
"""Golden vectors for the figure-3 scan-position engine (SURVEY.md 8f row 2), captured from the
UNMODIFIED reference function `simulate_imaging`
(figure_generation/line_sted_figure_3.py:76-273), read from $LSTED_REFERENCE_DIR or
baseline/_ref/ (tests/_reference_loader.py):
    python tests/golden/make_golden_fig3.py
The reference script calls main() at import and draws with matplotlib, so it is executed from
its source text with that last call left out and with `generate_figure` / `animate` replaced by
recorders -- the simulation code itself runs untouched.  Output (committed): fig3_frames.npz
 * every argument `simulate_imaging` hands to `generate_figure` for a few scan positions
   (first / one in the middle / last of every orientation; the last only for the cases at the
   script's own size), as float64 arrays,
 * sum and max of every array of EVERY drawn frame (so all positions are pinned),
 * the call counts (scan positions, camera exposures) the appendix table publishes
   (appendix.html:325-369);
and fig3_object_lines.npz: `object_u8`, the 8-bit test_object_lines.tif every case crops.
The committed copy of that image was read back from the stored frames (glow / excitation of
the rot-0 frames is the object times a constant; the 89-valued background filled the pixels
no stored excitation reaches) and reproduces every stored frame bit for bit.
"""
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from _reference_loader import load_reference, REFERENCE_DIR  # noqa: E402

ARRAYS = ('obj', 'excitation', 'glow', 'inst_sig', 'cum_sig', 'new_sig', 'reconstruction')


def load_figure3_namespace():
    """The reference script's globals, without running its main()."""
    load_reference()                      # installs the matplotlib stub and np_tif
    path = os.path.join(REFERENCE_DIR, 'line_sted_figure_3.py')
    with open(path) as f:
        src = f.read()
    assert src.rstrip().endswith('main()')
    src = src.rstrip()[:-len('main()')]
    ns = {'__name__': 'reference_figure_3', '__file__': path}
    plt = sys.modules['matplotlib.pyplot']
    if not hasattr(plt, 'figure'):
        plt.figure = lambda *a, **k: None
    exec(compile(src, path, 'exec'), ns)
    return ns


def capture(ns, *args, **kwargs):
    """Run the reference's simulate_imaging, recording what it would have drawn."""
    calls = []

    def recorder(filename, *a):
        rot = int(os.path.basename(filename).split('deg_')[0].split('_')[-1])
        calls.append(dict(rot=rot, which_pos=int(filename[-10:-4]),
                          arrays=[np.array(x, dtype=np.float64) for x in a[:7]],
                          pulses_delivered=a[7], camera_exposures=a[8]))
    ns['generate_figure'] = recorder
    ns['animate'] = lambda *a, **k: None
    stdout = sys.stdout
    sys.stdout = open(os.devnull, 'w')
    try:
        ns['simulate_imaging'](*args, **kwargs)
    finally:
        sys.stdout.close()
        sys.stdout = stdout
    return calls


CASES = {
    # name: (object crop, imaging_type, psf_width, R, num_orientations, pulses, pad)
    'small_descan_point': (48, 'descan_point', 10, 2, 1, 1, 10),
    'small_multipoint': (48, 'nondescan_multipoint', 10, 2, 1, 1, 10),
    'small_descan_line': (48, 'descan_line', 10, 2, 3, 1, 21),
    'small_rescan_line': (48, 'rescan_line', 10, 2, 3, 2, 21),
    'small_rescan_line_R1': (40, 'rescan_line', 9, 1, 2, 1, 18),
    'small_rescan_line_R3': (56, 'rescan_line', 13, 3, 2, 1, 25),
    # the script's own parameters (line_sted_figure_3.py:40-63), 1x1 field of view, R = 2
    'fig3_descan_line': (128, 'descan_line', 25, 2, 2, 1, 57),
    'fig3_rescan_line': (128, 'rescan_line', 25, 2, 2, 1, 57),
    'fig3_multipoint': (128, 'nondescan_multipoint', 25, 2, 1, 1, 25),
}


def lines_u8():
    return sys.modules['np_tif'].tif_to_array(os.path.join(REFERENCE_DIR, 'test_object_lines.tif'))


def make_object(ns, crop):
    obj = lines_u8() / 255 + 1e-6
    lo = (128 - crop) // 2
    return np.ascontiguousarray(obj[:, lo:lo + crop, lo:lo + crop])


def main():
    ns = load_figure3_namespace()
    store, meta = {}, {}
    for name, (crop, typ, width, R, n_or, pulses, pad) in CASES.items():
        obj = make_object(ns, crop)
        calls = capture(ns, obj, typ, width, R, n_or, pulses, pad, comparison_name=name)
        rots = sorted({c['rot'] for c in calls}, reverse=True)
        info = dict(crop=crop, imaging_type=typ, psf_width=width, R=R, num_orientations=n_or,
                    pulses_per_position=pulses, pad=pad, num_frames=len(calls), rotations=rots,
                    frames=[])
        sums = np.zeros((len(calls), len(ARRAYS), 2))
        for i, c in enumerate(calls):
            info['frames'].append([c['rot'], c['which_pos'], c['pulses_delivered'],
                                   c['camera_exposures']])
            for j, a in enumerate(c['arrays']):
                sums[i, j] = a.sum(), a.max()
        store[name + '/sums'] = sums
        for rot in rots:
            mine = [c for c in calls if c['rot'] == rot]
            picks = (mine[-1],) if name.startswith('fig3_') else (mine[0], mine[len(mine) // 2], mine[-1])
            for c in picks:
                for a, arr in zip(ARRAYS[1:], c['arrays'][1:]):
                    store['%s/%03d/%06d/%s' % (name, rot, c['which_pos'], a)] = arr
        meta[name] = info
        print(name, len(calls), 'frames')
    # the reference's own table (appendix.html:325-369): scan positions per method
    np.savez_compressed(os.path.join(HERE, 'fig3_frames.npz'), **store)
    np.savez_compressed(os.path.join(HERE, 'fig3_object_lines.npz'), object_u8=lines_u8())
    with open(os.path.join(HERE, 'fig3_frames.json'), 'w') as f:
        json.dump(meta, f, indent=0)


if __name__ == '__main__':
    main()
