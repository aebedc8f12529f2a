"""Local error metrics for the GPU parity checks: bound the error of every unit of work a kernel
owns, so that a fault in one CTA or one tile cannot hide in a whole-stack relative L2.

The engine splits its work so that a fault stays local:
  - a row CTA owns one orientation k and 2 * row_pairs_per_cta image rows;
  - a column CTA owns cols_per_cta bins of the row spectrum (x-frequencies), over all y; a fault
    there is a narrow band of x-frequencies, spread over every pixel in image space;
  - a tile of the overlap-save engine owns tile_out_y x tile_out_x output pixels.
Each metric below is measured per such unit.  For operator outputs (H, unnormalised H_t, the
noiseless field) of shape (K, Ny, Nx):
  orientation   relative L2 of each k on its own;
  peak          max |got - want| / RMS(want), per k;
  row group     sqrt(E_b / (R_b + R / n)) per (k, band of 2 * row_pairs_per_cta rows), E the error's
                energy, R the reference's, R / n its mean share per band (keeps nearly dark bands
                from dividing by zero);
  column block  the same ratio per (k, block of cols_per_cta bins) of the rfft along x of the error
                and of the reference, zero-padded to Lx (per tile on tiled handles, whose windows
                are Lx wide);
  tile          the same ratio per (k, output tile), tiled handles only.
For Richardson-Lucy estimates: the per-pixel |got - want| / (|want| + f * max|want|).

Bounds are multiples of eps * log2(Ly * Lx), eps = 2^-24 (fp32) or 2^-53 (fp64), so that they
scale with the transform length."""
from collections import namedtuple

import numpy as np

EPS = {32: 2.0 ** -24, 64: 2.0 ** -53}

# Bounds in units of eps * log2(Ly * Lx): 4x or more the worst value measured on one NVIDIA B200
# (1000 W power limit) over every case of the GPU parity suites and probes; the worst measured
# value and its case are beside each.  The lattice probes set the peak bound: their dark gaps
# lower RMS(want).
BOUND = {
    32: {'orientation': 2.0,    # 0.41  dark_fp32 noiseless (tiled)
         'peak': 64.0,          # 15.1  fixed_2048_centred_otf_fp32 lattice H_t
         'row group': 2.0,      # 0.44  dark_fp32 noiseless (tiled)
         'column block': 6.0,   # 1.30  w2160_row_plan2 H, H_t, noiseless (bins 1056-1059)
         'tile': 2.0,           # 0.37  dark_fp32 noiseless
         'estimate': 800.0},    # 198   dark_fp32 after 2 iterations
    64: {'orientation': 2.0,    # 0.43  fp64_fig2_runtime_dark H
         'peak': 64.0,          # 15.1  plan2160d_fp64 lattice H_t
         'row group': 2.0,      # 0.40  plan2160d_fp64 lattice H
         'column block': 6.0,   # 1.44  generic_fp64_PR1_3375 noiseless (bins 1124-1125)
         'tile': 1.0,           # 0.24  w2160_asym21_fp64 H
         'estimate': 512.0},    # 125   fp64_fig2_runtime_dark after 1 iteration
}

# f of the estimate metric: pixels far below the brightest one (the dark background of sparse
# objects) are judged against f * max|want| instead of their own value.  Without it the dark
# pixels of the bead objects dominate; on the CPU stand-in's dark object one fp32 RL step
# scores 63 units with f = 0 and 37 with f = 1e-3.
ESTIMATE_FLOOR = 1e-3

Geometry = namedtuple('Geometry', 'Ly Lx cols_per_cta row_pairs_per_cta tiles_y tiles_x '
                                  'tile_out_y tile_out_x')


def geometry(info):
    """The block geometry of a handle's info()."""
    return Geometry(info.Ly, info.Lx, info.cols_per_cta, info.row_pairs_per_cta,
                    info.tiles_y, info.tiles_x, info.tile_out_y, info.tile_out_x)


def unit(precision, geom):
    return EPS[precision] * np.log2(geom.Ly * geom.Lx)


def _tiles(shape, geom):
    """(y0, y1, x0, x1) of each output tile; the whole image on untiled handles."""
    Ny, Nx = shape
    if geom.tiles_y * geom.tiles_x <= 1:
        return [(0, Ny, 0, Nx)]
    return [(ty * geom.tile_out_y, min((ty + 1) * geom.tile_out_y, Ny),
             tx * geom.tile_out_x, min((tx + 1) * geom.tile_out_x, Nx))
            for ty in range(geom.tiles_y) for tx in range(geom.tiles_x)]


def _share_ratio(err_energy, ref_energy):
    """sqrt(E_b / (R_b + R / n)) over the last axis of per-unit energies."""
    n = ref_energy.shape[-1]
    return np.sqrt(err_energy / (ref_energy + ref_energy.sum(-1, keepdims=True) / n))


class LocalErrors:
    """Every local metric of `got` against `want` for one handle geometry.  `values[name]` is an
    array over units; `where[name](index)` names the unit of a flat index."""

    def __init__(self, got, want, geom, precision, estimate=False):
        got = np.asarray(got, np.float64)
        want = np.asarray(want, np.float64)
        want = want.reshape((-1,) + want.shape[-2:])
        got = got.reshape(want.shape)
        self.precision, self.geom, self.unit = precision, geom, unit(precision, geom)
        self.values, self.where = {}, {}
        err = got - want
        if estimate:
            a = np.abs(want)
            v = np.abs(err) / (a + ESTIMATE_FLOOR * a.max())
            self._add('estimate', v, lambda i: 'k = %d, pixel (%d, %d)' % np.unravel_index(i, v.shape))
            return
        K, Ny, Nx = want.shape
        e2, r2 = err ** 2, want ** 2
        self._add('orientation', np.sqrt(e2.sum((1, 2)) / r2.sum((1, 2))), lambda i: 'k = %d' % i)

        at = [np.unravel_index(np.argmax(np.abs(err[k])), (Ny, Nx)) for k in range(K)]
        peak = [abs(err[k][p]) for k, p in enumerate(at)] / np.sqrt(r2.mean((1, 2)))
        self._add('peak', peak, lambda k: 'k = %d, pixel (%d, %d)' % ((k,) + at[k]))

        band = 2 * geom.row_pairs_per_cta
        tiles = _tiles((Ny, Nx), geom)
        rows = []                       # (tile, first row of the band, last row)
        eb, rb = [], []
        for t, (y0, y1, x0, x1) in enumerate(tiles):
            for b in range(y0, y1, band):
                rows.append((t, b, min(b + band, y1) - 1))
                eb.append(e2[:, b:b + band, x0:x1].sum((1, 2)))
                rb.append(r2[:, b:b + band, x0:x1].sum((1, 2)))
        v = _share_ratio(np.stack(eb, 1), np.stack(rb, 1))
        tiled = len(tiles) > 1

        def row_unit(i):
            k, j = np.unravel_index(i, v.shape)
            t, b0, b1 = rows[j]
            return 'k = %d, %srows %d-%d' % (k, 'tile %d, ' % t if tiled else '', b0, b1)
        self._add('row group', v, row_unit)

        C = geom.cols_per_cta
        nbins = geom.Lx // 2 + 1
        nblocks = -(-nbins // C)
        ce, cr = [], []
        for (y0, y1, x0, x1) in tiles:
            assert x1 - x0 <= geom.Lx, (x1 - x0, geom.Lx)
            # spectral energy per bin, summed over y; one orientation at a time to bound memory
            fe = np.stack([(np.abs(np.fft.rfft(err[k, y0:y1, x0:x1], n=geom.Lx)) ** 2).sum(0)
                           for k in range(K)])
            fr = np.stack([(np.abs(np.fft.rfft(want[k, y0:y1, x0:x1], n=geom.Lx)) ** 2).sum(0)
                           for k in range(K)])
            pad = ((0, 0), (0, nblocks * C - nbins))
            ce.append(np.pad(fe, pad).reshape(K, nblocks, C).sum(2))
            cr.append(np.pad(fr, pad).reshape(K, nblocks, C).sum(2))
        v2 = _share_ratio(np.stack(ce, 1), np.stack(cr, 1)).reshape(K, -1)

        def col_unit(i):
            k, j = np.unravel_index(i, v2.shape)
            t, b = divmod(j, nblocks)
            return 'k = %d, %scolumn block %d (bins %d-%d)' % (
                k, 'tile %d, ' % t if tiled else '', b, b * C, min(b * C + C, nbins) - 1)
        self._add('column block', v2, col_unit)

        if tiled:
            te = np.stack([e2[:, y0:y1, x0:x1].sum((1, 2)) for (y0, y1, x0, x1) in tiles], 1)
            tr = np.stack([r2[:, y0:y1, x0:x1].sum((1, 2)) for (y0, y1, x0, x1) in tiles], 1)
            v3 = _share_ratio(te, tr)

            def tile_unit(i):
                k, t = np.unravel_index(i, v3.shape)
                y0, y1, x0, x1 = tiles[t]
                return 'k = %d, tile %d (rows %d-%d, columns %d-%d)' % (k, t, y0, y1 - 1, x0, x1 - 1)
            self._add('tile', v3, tile_unit)

    def _add(self, name, values, where):
        self.values[name] = np.asarray(values, np.float64).ravel()
        self.where[name] = where

    def bound(self, name):
        return BOUND[self.precision][name] * self.unit

    def worst(self):
        """{metric: (worst value, in units of eps * log2(Ly * Lx), its unit)}."""
        out = {}
        for name, v in self.values.items():
            i = int(np.argmax(v))
            out[name] = (v[i], v[i] / self.unit, self.where[name](i))
        return out

    def report(self, label):
        """One line with the worst value of every metric, so that each run logs its numbers."""
        return 'local %s (fp%d, Ly x Lx = %d x %d): %s' % (
            label, self.precision, self.geom.Ly, self.geom.Lx, '; '.join(
                '%s %.2e = %.3g u at %s' % (name, v, u, at)
                for name, (v, u, at) in self.worst().items()))

    def failures(self, label):
        """One message per metric whose bound fails, naming its worst unit."""
        out = []
        for name, v in self.values.items():
            bad = np.flatnonzero(v > self.bound(name))
            if bad.size:
                i = bad[np.argmax(v[bad])]
                out.append('%s: %s %s: %.2e > %.2e (%d of %d units over)' % (
                    label, name, self.where[name](i), v[i], self.bound(name), bad.size, v.size))
        return out


def local_errors(got, want, info, precision, estimate=False):
    return LocalErrors(got, want, info if isinstance(info, Geometry) else geometry(info),
                       precision, estimate)


def check_local(results):
    """Print the worst value of every metric of every (label, LocalErrors) pair, then assert
    every bound at once; the message names each failing unit."""
    for label, r in results:
        print(r.report(label))
    msgs = [m for label, r in results for m in r.failures(label)]
    assert not msgs, '\n'.join(msgs)
