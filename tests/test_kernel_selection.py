"""Which kernel instance runs each launch (dispatch.h: select_row / select_col), pinned on the
CPU replay.  The replay and the CUDA backend choose through the same functions, so the table
below is what the GPU runs for every case of test_gpu_dispatch_parity.py: a planner or
selection change that moves GPU dispatch fails here without a GPU.

Each row opens a replay handle with the case's shape, PSFs, precision, environment and options,
runs H, create_data and one RL iteration, and compares the logged (variant, geometry, TMA level)
of every row launch and (variant, geometry, CTAs per column block) of every column launch with
the table.  The expected choices follow from the selection rules:
  * rows run the 2160 plan when fast_path is on, Lx = 2160 and the column geometry has the
    plan's C (fp32 4, fp64 2); fp32 row kernels that index pixels (all but row_fwd) take the
    2048-wide geometry when Nx = 2048, Ny is even and the crop offset is 53 (g2048) or 0
    (centred real OTFs: g2048c); row_mid / row_final stage the spectra by tensor maps (fp32) at
    level row_tma, level 2 only where Nx * 4 is a multiple of 16;
  * columns run the 2160 plan for col_h / col_ht when Ly = 2160 and C is the plan's; centred
    real OTFs (point-symmetric PSFs) take the sub-block CTAs unless col_sub is off; fp32 with
    Ny = 2048 takes g2048 (crop offset 53) or g2048c (real OTFs);
  * generic col_h spreads the orientations of a block over min(148 / nxb, K, 3) CTAs on the
    replay (a B200 with one live handle; up to 3 CTAs per block) when 2 nxb <= 148 and K > 1."""
import ctypes

import numpy as np
import pytest

import emul_support
import test_gpu_dispatch_parity as parity
from rescan_line_sted_b200 import _lib

KINDS = ('row_fwd', 'row_inv_store', 'row_inv_sim', 'row_mid', 'row_final', 'col_otf', 'col_h', 'col_ht')
ROW_VARIANTS = ('generic', 'fast', 'row2', 'row_mid_dual')
COL_VARIANTS = ('generic', 'fast', 'fast_sub', 'ht_p2p')
GEOMS = ('runtime', 'g2048', 'g2048c')
LOG_INTS = 7        # emul.cpp: kind, variant, geometry, TMA level, real OTFs, grid, CTAs per block


def generic_rows():
    return {k: ('generic', 'runtime', 0) for k in KINDS[:5]}


def fast_rows(geom='runtime', tma=0, variant='fast'):
    t = {k: (variant, geom, 0) for k in KINDS[:5]}
    t['row_fwd'] = (variant, 'runtime', 0)
    t['row_mid'] = t['row_final'] = (variant, geom, tma)
    return t


def dual_rows():
    t = fast_rows('g2048c', 2)
    t['row_mid'] = ('row_mid_dual', 'runtime', 0)
    return t


def cols(variant='generic', geom='runtime', k_split=1):
    return {'col_h': (variant, geom, k_split), 'col_ht': (variant, geom, 1)}


def expect(rows, columns):
    return dict(rows, **columns)


GENERIC = expect(generic_rows(), cols())
GENERIC_SPLIT2 = expect(generic_rows(), cols(k_split=2))
FIG2_FP32 = expect(fast_rows('g2048c', 2), cols('fast_sub', 'g2048c'))
FIXED_2048 = expect(fast_rows('g2048', 2), cols('fast', 'g2048'))
FP64_FIG2 = expect(fast_rows(), cols('fast_sub'))

EXPECTED = {
    'fastrows_gencols_tma0': expect(fast_rows(), cols()),
    'fastrows_gencols_tma1': expect(fast_rows(tma=1), cols()),
    'fastrows_gencols_tma2': expect(fast_rows(tma=2), cols()),
    'fastrows_gencols_odd_2049': expect(fast_rows(tma=1), cols()),       # 2049 * 4 % 16 != 0
    'fastrows_gencols_fp64': expect(fast_rows(), cols()),
    'genrows_fastcols_2048c_sub0': expect(generic_rows(), cols('fast', 'g2048c')),
    'genrows_fastcols_2048c_sub1': expect(generic_rows(), cols('fast_sub', 'g2048c')),
    'genrows_fastcols_runtime_fp32': expect(generic_rows(), cols('fast_sub')),
    'genrows_fastcols_runtime_fp64': expect(generic_rows(), cols('fast_sub')),
    'fixed_2048_asym107': FIXED_2048,
    'fixed_2048_fig2_complex_otf': FIXED_2048,
    'fp64_fig2_sub0': expect(fast_rows(), cols('fast')),
    'fp64_fig2_sub1': FP64_FIG2,
    # the clip-per-term iteration updates the estimate elementwise: no row_final
    'fp64_fig2_exact_clip': {k: v for k, v in FP64_FIG2.items() if k != 'row_final'},
    'fp64_fig2_runtime_dark': FP64_FIG2,
    'fig2_row_plan2': expect(fast_rows(variant='row2'), cols('fast_sub', 'g2048c')),
    'fig2_row_dual': expect(dual_rows(), cols('fast_sub', 'g2048c')),
    'fig2_prefetch0': FIG2_FP32,
    'lx2160_genrows_fp32_C2': GENERIC,
    'lx2160_genrows_fp64_C1': GENERIC,
    'generic_fp32_C2': GENERIC_SPLIT2,            # 7 column blocks
    'generic_fp32_C1_6075': GENERIC_SPLIT2,       # 55 column blocks: 148 // 55 = 2
    'generic_fp32_PR1_7200': GENERIC,
    'generic_fp64_C1': GENERIC_SPLIT2,
    'generic_fp64_PR1_3375': GENERIC,
    'generic_fp32_3125': GENERIC,
    'generic_fp64_3125': GENERIC,
    'radix_tail_fp32_32x64': GENERIC_SPLIT2,
    'radix_tail_fp32_128': GENERIC_SPLIT2,
    'radix_tail_fp64_64x32': GENERIC_SPLIT2,
    'radix_tail_fp64_128': GENERIC_SPLIT2,
    'fast_path0_2160_asym': GENERIC,
    'fast_path0_2160_fig2': GENERIC,
}

# the reference's frame size (128^2, K = 10, 25 column blocks): 3 CTAs per block, or 1 with the
# option off; the default 2048^2 fp32 figure-2 case
EXTRA = {
    'k_split_128': (parity.case((128, 128), 'asym107', 32, (192, 192, 4, 2), K=10),
                    expect(generic_rows(), cols(k_split=3))),
    'k_split_off_128': (parity.case((128, 128), 'asym107', 32, (192, 192, 4, 2), K=10,
                                    options=[('k_split', 0)]), GENERIC),
    'default_2048_fig2': (parity.case((2048, 2048), 'fig2', 32, (2160, 2160, 4, 2)), FIG2_FP32),
}


@pytest.fixture(scope='module')
def lib():
    return emul_support.emulator_library()


def dispatch_log(lib, first):
    n = lib.cdll.emul_dispatch_log(first, None, 0)
    buf = (ctypes.c_int * (LOG_INTS * max(n - first, 1)))()
    lib.cdll.emul_dispatch_log(first, buf, n - first)
    return np.array(buf[:LOG_INTS * (n - first)]).reshape(-1, LOG_INTS)


def choices(log):
    """{kind: {(variant, geometry, TMA level or CTAs per column block)}} of the logged launches."""
    seen = {}
    for kind, variant, geom, tma, _, _, k_split in log:
        name = KINDS[kind]
        if name.startswith('row'):
            c = (ROW_VARIANTS[variant], GEOMS[geom], int(tma))
        else:
            c = (COL_VARIANTS[variant], GEOMS[geom], int(k_split))
        seen.setdefault(name, set()).add(c)
    return seen


def open_replay(lib, c, monkeypatch):
    """A replay handle opened like the GPU test's handle (test_gpu_dispatch_parity.open_handle)."""
    for name, value in c.env:
        monkeypatch.setenv(name, value)
    h = _lib.DeconvHandle(lib, parity.make_psfs(c.psf, c.K), c.shape, precision=c.precision)
    for name, _ in c.env:
        monkeypatch.delenv(name)
    info = h.info()
    assert (info.Ly, info.Lx, info.cols_per_cta, info.row_pairs_per_cta) == c.info
    for name, value in c.options:
        h.set_option(name, value)
    return h


def run_case(lib, c, monkeypatch):
    """Runs H, create_data and one iteration; returns the choices of these launches."""
    h = open_replay(lib, c, monkeypatch)
    first = lib.cdll.emul_dispatch_log(0, None, 0)
    x = parity.make_object(c.shape, c.obj)
    h.H(x)
    h.create_data(x, 100.0 * x.size, 3)
    h.iterate(1)
    h.close()
    return choices(dispatch_log(lib, first))


def test_table_covers_every_gpu_dispatch_case():
    assert sorted(EXPECTED) == sorted(parity.CASES)


@pytest.mark.parametrize('name', sorted(EXPECTED) + sorted(EXTRA))
def test_kernel_choice(lib, name, monkeypatch):
    c, want = (parity.CASES[name], EXPECTED[name]) if name in EXPECTED else EXTRA[name]
    assert run_case(lib, c, monkeypatch) == {k: {v} for k, v in want.items()}


def test_default_2048_fig2_against_oracle(lib, monkeypatch):
    """The headline case on the replay, through the instances the GPU runs (RowGeom2048c with
    tensor-map staging, sub-block ColGeom2048c columns): H, unnormalised H_t and two RL
    iterations from the oracle's noise, against the fp64 oracle."""
    c = EXTRA['default_2048_fig2'][0]
    h = open_replay(lib, c, monkeypatch)
    first = lib.cdll.emul_dispatch_log(0, None, 0)
    try:
        x, y, B, Hx, Hty, noiseless, noisy, est = parity.oracle_results(c.shape, c.psf, c.K, c.obj)
        err = {'H': parity.rel_l2(h.H(x), Hx), 'Ht': parity.rel_l2(h.Ht(y, False), Hty)}
        h.create_data(x, B, 3)
        for k in range(c.K):
            h.set(_lib.NOISY, k, noisy[k])
        for n in (1, 2):
            h.iterate(1)
            err['iter%d' % n] = parity.rel_l2(h.get(_lib.ESTIMATE), est[n - 1])
    finally:
        h.close()
    print('measured replay default_2048_fig2: ' + ', '.join('%s %.2e' % kv for kv in err.items()))
    assert choices(dispatch_log(lib, first)) == {k: {v} for k, v in FIG2_FP32.items()}
    assert err['H'] < 1e-5 and err['Ht'] < 1e-5
    assert err['iter1'] < 1e-4 and err['iter2'] < 1e-4
