#!/usr/bin/env python3
"""Headline benchmark: simulated rescan-line-STED frames/s at 2048^2.

One step = one frame(N_iter) of BASELINE.json config 4 (SURVEY.md 8d):
    create_data_from_object (K forward convolutions + Poisson)
    + H_t_normalization + N_iter Richardson-Lucy iterations,
on a synthetic 2048^2 object (astronaut tiled 16x16), K = 16 line
orientations of the figure-2 '2p0x_lr' rescan PSF (107^2), fp32.

  python bench.py [--gpus N] [--steps K] [--warmup W]       this repo (CUDA)
  python bench.py --impl reference ...                      CPU reference arm
  python bench.py ... --dump-outputs DIR                    + the last timed frame as .npy

With N > 1 (torchrun) every rank simulates and deconvolves its own frames
(independent frames = the reference's own unit of parallel work: figure 2
runs 24 deconvolvers x 4 images); no data-path collective, weak scaling.
The same line then carries an `orientation_sharded` record: ONE frame with its
K orientations split over the N GPUs (strong scaling, the per-iteration sum
fused into the column kernel over NVLink peer memory), its speed-up over the
rank-local unsharded frame and the rel-L2 between the two estimates.
Prints ONE JSON line on rank 0.

`e2e` goes through the reference-facing API: line_sted_tools.Deconvolver --
create_data_from_object(host object) + 64 x iterate() + read of `.estimate`.
The reference arm runs the UNMODIFIED reference module from baseline/_ref/
(a git-ignored copy of the reference's figure_generation directory, where one
was placed; `kind: "reference"`), or the oracle port when that copy is absent
(`kind: "port"`).

--dump-outputs DIR writes what the timed frame hands its caller, from the last
timed step: DIR/estimate.npy (1, N, N) and DIR/noisy_measurement.npy /
DIR/noiseless_measurement.npy (K, N, N), in the engine's precision (float32 or
float64).  The files take at most 64 MB: an array too large for its share (half
for the estimate, a quarter for each measurement) is replaced by the same fixed,
seeded sample of pixels of every plane (K, P); at the defaults that is the two
measurements.  Inputs and seeds depend only on the arguments, so two
builds can be compared output for output.  Nothing is written to the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # the tree may be read-only; leave it as it is
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FIG2_2P0X_LR = dict(excitation_brightness=0.21672180512595912,
                    depletion_brightness=11.766131198861775,
                    steps_per_excitation_psf_width=25, pulses_per_position=5)
EMISSION_2P0X_LR = 3.0227


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='cuda', choices=['cuda', 'reference'])
    ap.add_argument('--size', type=int, default=2048)
    ap.add_argument('--orientations', type=int, default=16)
    ap.add_argument('--iterations', type=int, default=64)
    ap.add_argument('--precision', default='fp32', choices=['fp32', 'fp64'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-fp64', action='store_true', help='skip the fp64 companion figure')
    ap.add_argument('--no-sweep', action='store_true', help='skip the config-3 PSF sweep record')
    ap.add_argument('--shard', default='frames', choices=['frames', 'orientations'],
                    help='N>1: independent frames per GPU (weak scaling, no collective) or the '
                         'K orientations of every frame split over the GPUs (strong scaling, one '
                         'NCCL all-reduce per RL iteration)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step to DIR/<name>.npy (rank 0)')
    return ap.parse_args()


# ---------------------------------------------------------------------------
# Workload (host-side, one-off, outside every timed region)
# ---------------------------------------------------------------------------
def rotate_psf(x, degrees):
    """Orientation step of the caller (line_sted_figure_2.py:264-272)."""
    from scipy.ndimage import rotate
    if degrees == 0:
        return x
    if degrees == 90:
        return np.rot90(np.squeeze(x)).reshape(x.shape)
    return np.clip(rotate(x, angle=degrees, axes=(1, 2), reshape=False),
                   0, 1.1 * x.max())


def orientation_psfs(base, K):
    unit = base / base.sum()
    return [1 / K * EMISSION_2P0X_LR * rotate_psf(unit, a)
            for a in np.arange(0, 180, 180 / K)]


def synthetic_object(N):
    """O1 of SURVEY.md 8d: the 128^2 astronaut target tiled to N x N."""
    tile = np.load(os.path.join(ROOT, 'tests', 'golden', 'fig2_2p0x_lr.npz'))['object_u8']
    reps = (N + 127) // 128
    return np.ascontiguousarray(
        np.tile(tile, (1, reps, reps))[:, :N, :N].astype(np.float64))


def total_brightness(N):
    return 5e10 * (N / 128.0) ** 2


# ---------------------------------------------------------------------------
# Clock sampling during the timed region
# ---------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled through NVML (same data as the
    nvidia-smi clocks line of B200_PROFILING.md, without spawning a process
    that stalls the driver) every 20 ms from a thread."""
    REASONS = (('hw_slowdown', 0x8), ('sw_thermal_slowdown', 0x20),
               ('hw_thermal_slowdown', 0x40), ('sw_power_cap', 0x4))

    def __init__(self, device):
        self.device, self.rows, self.thread = device, [], None
        self.running, self.error = False, None
        self.t0 = self.t1 = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            index = self.device
            if visible:
                ids = [v for v in visible.split(',') if v.strip()]
                if all(v.strip().isdigit() for v in ids) and self.device < len(ids):
                    index = int(ids[self.device])
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as exc:  # noqa: BLE001
            self.error = repr(exc)
            return
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _loop(self):
        nv = self.nvml
        while self.running:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            except Exception:  # noqa: BLE001
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                except Exception:  # noqa: BLE001
                    reasons = 0
            self.rows.append((time.perf_counter(), float(mhz), int(reasons)))
            time.sleep(0.02)

    def window(self, t0, t1):
        """Only samples taken inside [t0, t1] (the timed region) count."""
        self.t0, self.t1 = t0, t1

    def stop(self):
        if self.thread is None:
            return {'sm_mhz': None, 'sm_max_mhz': None,
                    'reasons': ['NVML unavailable: %s' % self.error]}
        self.running = False
        self.thread.join(timeout=1.0)
        rows = [r for r in self.rows
                if self.t0 is None or self.t0 <= r[0] <= self.t1 + 0.03] or self.rows[-1:]
        sm = [r[1] for r in rows]
        bits = 0
        for r in rows:
            bits |= r[2]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(n for n, b in self.REASONS if bits & b),
                'samples': len(sm)}


# ---------------------------------------------------------------------------
# CPU reference arm / cpu_baseline (the only place bench.py runs oracle/ or baseline/_ref)
# ---------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')


def load_reference_module():
    """The unmodified reference `line_sted_tools` from baseline/_ref (None when absent).
    matplotlib is not installed in the image; the module imports it at the top and never
    uses it, so an empty stand-in module goes into sys.modules (no source change)."""
    path = os.path.join(REF_DIR, 'line_sted_tools.py')
    if not os.path.isfile(path):
        return None
    import importlib.util
    import types
    import warnings
    for name in ('matplotlib', 'matplotlib.pyplot'):
        if name not in sys.modules:
            try:
                __import__(name)
            except ImportError:
                sys.modules[name] = types.ModuleType(name)
    sys.path.insert(0, REF_DIR)          # its own `import np_tif`
    try:
        spec = importlib.util.spec_from_file_location('reference_line_sted_tools', path)
        mod = importlib.util.module_from_spec(spec)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            spec.loader.exec_module(mod)
    finally:
        sys.path.remove(REF_DIR)
    return mod


def host_cores():
    """All the cores of the box, also under torchrun (which may narrow the affinity)."""
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def reference_psfs(ref, K):
    """The benchmark PSFs by the reference's own psf_report (+ the caller's rotate)."""
    if ref is None:
        from oracle import line_sted_oracle as orc
        return orc.benchmark_psfs(K)
    base = ref.psf_report('line', verbose=False, **FIG2_2P0X_LR)['psfs']['rescan_sted']
    return orientation_psfs(base, K)


def cpu_reference_frame(args, obj, psfs, ref, workers, warmup, steps):
    """Times the reference Deconvolver exactly as figure 2 drives it
    (line_sted_figure_2.py:40-56): create_data_from_object, then iterate() calls -- the first
    one also builds the estimate and H_t_normalization (ref:521-522, :589-593) -- on the
    full-size workload with scipy.fft workers = all cores (a context manager around the
    unmodified code).  frame(n) = forward + first iterate() + (n-1) x mean later iterate()."""
    import tempfile
    import warnings
    import scipy.fft
    N = obj.shape[-1]
    if ref is not None:
        make = lambda: ref.Deconvolver(psfs, output_prefix=tempfile.mkdtemp() + os.sep, verbose=False)
        kind = 'reference'
    else:
        from oracle import line_sted_oracle as orc
        make = lambda: orc.Deconvolver(psfs, engine='scipy')
        kind = 'port'
    with scipy.fft.set_workers(workers), warnings.catch_warnings():
        warnings.simplefilter('ignore')
        d = make()
        t0 = time.perf_counter()
        d.create_data_from_object(obj, total_brightness=total_brightness(N), random_seed=0)
        t_forward = time.perf_counter() - t0
        t0 = time.perf_counter()
        d.iterate()
        t_first = time.perf_counter() - t0
        for _ in range(warmup):
            d.iterate()
        its = []
        for _ in range(steps):
            t0 = time.perf_counter()
            d.iterate()
            its.append(time.perf_counter() - t0)
    t_iter = float(np.mean(its))
    n = args.iterations
    frame_s = t_forward + t_first + max(0, n - 1) * t_iter
    sample = ('%s Deconvolver at full size (%d^2, K=%d, float64), scipy.fft workers=%d: '
              'create_data_from_object %.2f s, first iterate() (incl. H_t_normalization) %.2f s, '
              '%d timed iterate() calls %.3f s each; frame(%d) = forward + first + %d x iterate '
              '(EXTRAPOLATED from the timed calls, %.0f s)'
              % ('unmodified reference' if ref is not None else 'oracle port of the reference',
                 N, len(psfs), workers, t_forward, t_first, steps, t_iter, n, n - 1, frame_s))
    return {'kind': kind, 'frame_s': frame_s, 'forward_s': t_forward, 'first_iterate_s': t_first,
            'iteration_s': t_iter, 'sample': sample, 'cores': workers}


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return                      # one CPU process: the other ranks exit without work
    workers = host_cores()
    ref = load_reference_module()
    N, K = args.size, args.orientations
    psfs = reference_psfs(ref, K)
    cpu = cpu_reference_frame(args, synthetic_object(N), psfs, ref, workers,
                              max(0, args.warmup - 1), max(1, args.steps))
    value = 1.0 / cpu['frame_s']
    print(json.dumps({
        'impl': 'reference', 'metric': 'frames_per_sec', 'value': value, 'unit': 'frames/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': cpu['frame_s'] * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(args),
        'cpu_baseline': {'value': value, 'unit': 'frames/s', 'cores': cpu['cores'],
                         'kind': cpu['kind'], 'sample': cpu['sample']},
        'note': 'one CPU process on rank 0 whatever --gpus says: compare it with the N=1 line',
        'e2e': {'value': value, 'unit': 'frames/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0}}))


def workload_config(args):
    return {'workload': 'config 4: synthetic %d^2 object (astronaut tiled), %d line orientations '
                        '(fig-2 2p0x_lr rescan PSF 107^2), Poisson noise + %d RL iterations '
                        '= frame(%d)' % (args.size, args.orientations, args.iterations,
                                         args.iterations),
            'size': args.size, 'orientations': args.orientations,
            'rl_iterations': args.iterations, 'psf_side': 107,
            'sharding': ('independent frames per GPU (no collective)' if args.shard == 'frames'
                         else 'orientations of each frame split over the GPUs, one NCCL all-reduce '
                              'of the Fourier-domain partial H_t sum per RL iteration'),
            'cache': 'working set (K measurements + K spectra + K OTFs, >1 GB) exceeds the '
                     '126 MB L2; no explicit flush'}


# ---------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------
def measured_peak():
    peaks_file = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(peaks_file):
        with open(peaks_file) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_facts(precision, N, K):
    """Per-launch DRAM bytes and pipe utilisation of the four iteration kernels from the
    committed `ncu --set full` capture of this workload (profiles/, newest round first)."""
    if precision != 'fp32' or N != 2048 or K != 16:
        return None
    for name in ('r02_dram_traffic.json', 'r01_dram_traffic.json'):
        path = os.path.join(ROOT, 'profiles', name)
        if os.path.isfile(path):
            with open(path) as f:
                t = json.load(f)
            t['_file'] = 'profiles/' + name
            return t
    return None


DUMP_BYTES = 63 * 10 ** 6          # array data of --dump-outputs: 64 MB with room for the headers


def dump_outputs(h, out_dir, dtype):
    """What one frame hands its caller: the estimate (up to half of DUMP_BYTES whole) and the K
    noisy / noiseless measurements (a quarter each).  An array that does not fit its share is
    stored as the same seeded sample of pixel positions of every plane.  `dtype` is the
    engine's precision, so nothing is rounded on the way out."""
    from rescan_line_sted_b200 import _lib
    os.makedirs(out_dir, exist_ok=True)
    n = h.Ny * h.Nx
    item = np.dtype(dtype).itemsize
    for name, which, planes, share in (('estimate', _lib.ESTIMATE, 1, DUMP_BYTES // 2),
                                       ('noisy_measurement', _lib.NOISY, h.K, DUMP_BYTES // 4),
                                       ('noiseless_measurement', _lib.NOISELESS, h.K, DUMP_BYTES // 4)):
        if planes * n * item <= share:
            out = np.stack([h.get(which, k)[0] for k in range(planes)]).astype(dtype)
        else:
            pixels = np.sort(np.random.default_rng(0).choice(n, share // (planes * item), replace=False))
            out = np.stack([h.get(which, k).reshape(-1)[pixels] for k in range(planes)]).astype(dtype)
        np.save(os.path.join(out_dir, name + '.npy'), out)


def time_frames(h, frame, seeds, barrier):
    barrier()
    h.timer_start()
    for s in seeds:
        frame(s)
    ms = h.timer_stop()
    barrier()
    return ms


def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    N, K, n_iter = args.size, args.orientations, args.iterations

    if args.impl == 'reference':
        run_reference_arm(args)
        return

    os.environ['LSTED_DEVICE'] = str(local_rank)
    os.environ['LSTED_PRECISION'] = args.precision
    from rescan_line_sted_b200 import _lib, line_sted_tools as st
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    # PSFs through the product's own PSF path (GPU): psf_report + on-device orientation step.
    from rescan_line_sted_b200 import orientations
    base = st.psf_report('line', verbose=False, **FIG2_2P0X_LR)['psfs']['rescan_sted']
    psfs = orientations.line_orientation_psfs(base, K, EMISSION_2P0X_LR)
    obj_host = synthetic_object(N)
    brightness = total_brightness(N)
    prec_bits = 32 if args.precision == 'fp32' else 64

    lib = _lib.get()
    by_orientation = args.shard == 'orientations' and world > 1
    if by_orientation:
        from rescan_line_sted_b200 import sharded
        sd = sharded.OrientationShardedDeconvolver(
            st._stack_psfs(psfs), (N, N), precision=prec_bits, device=local_rank)
        h = sd.handle
    else:
        h = _lib.DeconvHandle(lib, st._stack_psfs(psfs), (N, N), precision=prec_bits,
                              device=local_rank)
    jobs = 1 if by_orientation else world   # frames in flight across the node
    info = h.info()
    pinned_in = _lib.pinned_empty((1, N, N))
    pinned_in[...] = obj_host

    def frame_on(handle):
        def frame(seed):
            handle.set_option('forget_normalization', 1)
            handle.simulate(brightness, seed)        # (restarts the estimate from ones)
            handle.iterate(n_iter)
        return frame
    frame_resident = frame_on(h)

    def barrier():
        h.sync()
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        import torch
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing (headline `value`) ----
    seed0 = 0 if by_orientation else 7919 * rank
    h.upload_object(pinned_in)
    sampler = ClockSampler(local_rank)
    sampler.start()     # before the warm-up: nvidia-smi start-up stalls the driver briefly
    for w in range(args.warmup):
        frame_resident(1000 + w)
    barrier()
    t_begin = time.perf_counter()
    ms_total = time_frames(h, frame_resident, [s + 1 + seed0 for s in range(args.steps)], barrier)
    sampler.window(t_begin, time.perf_counter())
    if args.dump_outputs and rank == 0:
        dump_outputs(h, args.dump_outputs, np.float32 if args.precision == 'fp32' else np.float64)
    # Same K steps again with a CUDA-event pair around every launch (costs a few
    # microseconds of stream time per launch, so it is kept out of `value`): the
    # per-kernel durations behind `roofline` and `kernels`.
    h.set_option('profile', 1)
    h.profile(reset=True)
    for s in range(args.steps):
        frame_resident(s + 1 + seed0)
    prof = h.profile(reset=True)
    h.set_option('profile', 0)
    clocks = sampler.stop()
    ms_total = max_over_ranks(ms_total)
    ms_step = ms_total / args.steps
    value = jobs * 1000.0 / ms_step

    # ---- end-to-end through the reference-facing API (line_sted_figure_2.py:40-56) ----
    # host object (pinned) -> Deconvolver.create_data_from_object -> n_iter x iterate() -> .estimate
    h2d = int(pinned_in.nbytes)
    if by_orientation:
        pinned_out = _lib.pinned_empty((1, N, N))

        def frame_e2e(seed):
            h.upload_object(pinned_in)
            frame_resident(seed)
            h.get_into(_lib.ESTIMATE, 0, pinned_out)
            return pinned_out
        api = 'DeconvHandle of the orientation-sharded deconvolver (upload_object, simulate, iterate, get)'
    else:
        d = st.Deconvolver(psfs, output_prefix=os.path.join(tempfile.gettempdir(), 'lsted_bench_%d_' % rank),
                           verbose=False)
        d._handle, d._shape = h, (1, N, N)          # share the bench handle (OTFs already built)
        d._psf_key = tuple(id(p) for p in d.psfs)

        def frame_e2e(seed):
            d.num_iterations = 0
            d.create_data_from_object(pinned_in, total_brightness=brightness, random_seed=seed)
            for _ in range(n_iter):
                d.iterate()
            return d.estimate                        # D2H, fresh float64 array
        api = ('line_sted_tools.Deconvolver: create_data_from_object(host float64 object, pinned) '
               '+ %d x iterate() + read of .estimate' % n_iter)
    for w in range(min(2, args.warmup)):
        est = frame_e2e(2000 + w)
    barrier()
    t0 = time.perf_counter()
    h.timer_start()
    for s in range(args.steps):
        est = frame_e2e(s + 1)
    h.sync()
    wall = (time.perf_counter() - t0) * 1e3
    ms_e2e = max(h.timer_stop(), wall)
    barrier()
    ms_e2e = max_over_ranks(ms_e2e) / args.steps
    est = np.array(est)
    d2h = int(est.nbytes)
    if not np.isfinite(est).all() or est.min() < 0:
        raise RuntimeError('bench produced a non-finite estimate')

    # ---- N > 1: the same frame with its orientations split over the GPUs ----
    orientation_record = None
    if world > 1 and not by_orientation and K >= world:
        from rescan_line_sted_b200 import sharded
        sd = sharded.OrientationShardedDeconvolver(
            st._stack_psfs(psfs), (N, N), precision=prec_bits, device=local_rank)
        hs = sd.handle
        hs.upload_object(pinned_in)
        frame_sharded = frame_on(hs)
        for w in range(args.warmup):
            frame_sharded(1000 + w)
        ms_sh = max_over_ranks(time_frames(hs, frame_sharded,
                                           [s + 1 for s in range(args.steps)], barrier)) / args.steps
        # parity, witnessed in the driver's own run: same seed -> same Poisson field (keyed by
        # global orientation and pixel); compare with the rank-local unsharded frame
        frame_sharded(4242)
        frame_resident(4242)
        e_sh, e_1 = hs.get(_lib.ESTIMATE), h.get(_lib.ESTIMATE)
        rel = float(np.linalg.norm(e_sh - e_1) / np.linalg.norm(e_1))
        rel = max_over_ranks(rel)
        orientation_record = {
            'frames_per_sec': 1000.0 / ms_sh, 'ms_per_frame': ms_sh,
            'speedup_vs_one_gpu': ms_step / ms_sh, 'efficiency': ms_step / ms_sh / world,
            'rel_l2_vs_unsharded': rel, 'rel_l2_tolerance': 2e-4,
            'reduction': 'NVLS: multimem.ld_reduce / multimem.st through the NVSwitch (CUDA multicast object)'
                         if getattr(sd, 'nvls', False)
                         else 'fused into the column kernel over NVLink peer memory (P2P)' if sd.p2p
                         else 'ncclAllReduce of the Fourier-domain partial sum',
            'orientations_per_gpu': sd.k1 - sd.k0}
        sd.close()

    # ---- fp64-vs-fp64 companion figure (the tolerance-validation mode) ----
    fp64_record = None
    if args.precision == 'fp32' and not by_orientation and not args.no_fp64:
        h64 = _lib.DeconvHandle(lib, st._stack_psfs(psfs), (N, N), precision=64, device=local_rank)
        h64.upload_object(pinned_in)
        f64 = frame_on(h64)
        f64(1)
        n64 = max(1, min(3, args.steps))
        ms64 = max_over_ranks(time_frames(h64, f64, [s + 2 + seed0 for s in range(n64)], barrier)) / n64
        fp64_record = {'value': jobs * 1000.0 / ms64, 'unit': 'frames/s', 'ms_per_step': ms64,
                       'steps': n64, 'dtype': 'f64',
                       'note': 'same frame(%d) with the engine in fp64 (the reference\'s dtype)' % n_iter}
        h64.close()

    # ---- config 3 (SURVEY 8d): the 64-point PSF sweep, points dealt over the GPUs ----
    sweep_record = None
    if not args.no_sweep and not by_orientation:
        sys.path.insert(0, os.path.join(ROOT, 'scripts'))
        import sweep_times
        sweep_record = sweep_times.sweep_benchmark(rank, world, dist, repeats=3, big=16)
        sweep_record['note'] = ('psf_report_batch (one fused launch per rank: illumination, in-kernel '
                                'lmdif width fits, rescan PSF, doses), points dealt round-robin over '
                                'the GPUs, reports gathered once; wall clock, max over ranks')

    # ---- config 2 (the reference's own 128^2 frames) and the figure-3 scan engine, N = 1 ----
    config2_record = scan_record = None
    if world == 1 and not args.no_sweep:
        sys.path.insert(0, os.path.join(ROOT, 'scripts'))
        import config2_times
        import scan_times
        config2_record = config2_times.bench_record()
        scan_record = scan_times.bench_record()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (live CUDA-event timings) ----
    peak, peak_src = measured_peak()
    elem = 4 if args.precision == 'fp32' else 8
    A = elem * N * N
    K_total = K
    if by_orientation:
        K = sd.k1 - sd.k0       # per-GPU accounting: this rank's orientations
    total_kernel_ms = sum(v[0] for v in prof.values())
    launches = int(sum(v[1] for v in prof.values()))
    dom = max(prof, key=lambda k: prof[k][0])
    dom_ms, dom_n = prof[dom]
    kernels = {k: {'ms_per_step': v[0] / args.steps, 'launches_per_step': v[1] / args.steps,
                   'avg_ms': v[0] / v[1], 'share': v[0] / total_kernel_ms if total_kernel_ms else 0.0}
               for k, v in prof.items() if v[1]}
    # The iteration is one unit of (K+4)A bytes spread over its four launches:
    it_ms = sum(prof[k][0] for k in ('col_h', 'row_mid', 'col_ht', 'row_final')) / (
        args.steps * n_iter)
    step_bytes = (2 * K + 2 + n_iter * (K + 4)) * A
    roofline = {
        'bound': 'hbm', 'unit': 'GB/s', 'peak': peak, 'peak_source': peak_src,
        'kernel': dom, 'kernel_share_of_step': dom_ms / total_kernel_ms,
        'kernel_avg_ms': dom_ms / max(1, dom_n),
        'iteration_avg_ms': it_ms,
        'achieved': (K + 4) * A / (it_ms * 1e-3) / 1e9,
        'algorithmic_bytes': (K + 4) * A,
        'traffic': None,
        'note': 'achieved = (K+4)*A algorithmic bytes of one RL iteration / the summed average '
                'durations of its 4 launches (col_h,row_mid,col_ht,row_final).  The binding '
                'resources are the FP32 and shared-memory pipes (FFT butterflies), not HBM: '
                'fp32_pipe_frac / smem_pipe_frac / dram_frac below, DESIGN.md section 4',
    }
    facts = ncu_facts(args.precision, N, K_total) if not by_orientation else None
    if facts:
        names = ('col_h', 'row_mid', 'col_ht', 'row_final')
        traffic = sum(facts[k]['dram_bytes_read'] + facts[k]['dram_bytes_write'] for k in names)
        roofline['traffic'] = traffic
        roofline['traffic_source'] = facts.get('_source', facts['_file'])
        # real DRAM traffic of the iteration / its live duration / the measured copy peak
        roofline['dram_frac'] = traffic / (it_ms * 1e-3) / 1e9 / peak
        if all('fma_pipe_pct' in facts[k] for k in names):
            # time-weighted ncu pipe utilisation of the four launches (captured durations)
            tt = sum(facts[k]['duration_us'] for k in names)
            roofline['fp32_pipe_frac'] = sum(facts[k]['fma_pipe_pct'] * facts[k]['duration_us']
                                             for k in names) / tt / 100.0
            roofline['smem_pipe_frac'] = sum(facts[k]['l1tex_pct'] * facts[k]['duration_us']
                                             for k in names) / tt / 100.0
            roofline['binding'] = 'fp32 + shared-memory pipes (see fp32_pipe_frac, smem_pipe_frac)'
    roofline['frac'] = roofline['achieved'] / peak
    roofline['step_achieved'] = step_bytes / (ms_step * 1e-3) / 1e9
    roofline['step_frac'] = roofline['step_achieved'] / peak

    cfg = workload_config(args)
    cfg['e2e_api'] = api
    line = {
        'metric': 'frames_per_sec', 'value': value, 'unit': 'frames/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step,
        'higher_is_better': True, 'scaling': 'strong' if by_orientation else 'weak',
        'vs_baseline': None,
        'dtype': 'f32' if args.precision == 'fp32' else 'f64', 'data': 'synthetic',
        'config': cfg,
        'e2e': {'value': jobs * 1000.0 / ms_e2e, 'unit': 'frames/s',
                'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': ms_e2e},
        'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline, 'kernels': kernels,
        'rl_iterations_per_sec': jobs * n_iter * 1000.0 / ms_step,
        'geometry': {'Ly': info.Ly, 'Lx': info.Lx, 'cols_per_cta': info.cols_per_cta,
                     'row_pairs_per_cta': info.row_pairs_per_cta,
                     'device_bytes': int(info.device_bytes)},
    }
    extra = {}
    if fp64_record:
        extra['fp64'] = fp64_record
    if sweep_record:
        extra['config3_sweep'] = sweep_record
    if config2_record:
        extra['config2'] = config2_record
    if scan_record:
        extra['scan_engine'] = scan_record
    if orientation_record:
        line['orientation_sharded'] = orientation_record
    if extra:
        line['extra'] = extra
    if world == 1 and not args.no_cpu_baseline:
        ref = load_reference_module()
        cpu = cpu_reference_frame(args, obj_host, reference_psfs(ref, K_total), ref,
                                  host_cores(), 0, 1)
        line['cpu_baseline'] = {'value': 1.0 / cpu['frame_s'], 'unit': 'frames/s',
                                'cores': cpu['cores'], 'kind': cpu['kind'],
                                'sample': cpu['sample']}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
