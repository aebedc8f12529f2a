"""Frames/s of the reference's frame loop with numpy arrays against CUDA tensors.

The workload of bench.py (2048^2 synthetic object, K = 16 line orientations of the
figure-2 '2p0x_lr' rescan PSF, fp32 engine): create_data_from_object + 64 x
iterate() + a read of the estimate, through line_sted_tools.Deconvolver,
  numpy    host float64 object (pinned), `.estimate` (D2H, float64 array), as bench's e2e;
  tensor   float32 CUDA tensor object, `Deconvolver.tensor('estimate', float32)`;
  resident the same frame with the object already staged and no read (bench's headline).
Then one H and one H_t of a float32 tensor against a numpy array.  The arms alternate
in one process, `--rounds` times; the median of each is printed with the card's name
and power limit read in the same run.

  python scripts/device_io_times.py [--steps 5] [--rounds 3] [--iterations 64]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader',
                        '-i', '0'], capture_output=True, text=True)
    return q.stdout.strip() or 'unknown (nvidia-smi: %s)' % q.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--size', type=int, default=2048)
    ap.add_argument('--orientations', type=int, default=16)
    ap.add_argument('--iterations', type=int, default=64)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    args = ap.parse_args()
    N, K, n_iter = args.size, args.orientations, args.iterations
    os.environ['LSTED_PRECISION'] = 'fp32'
    import torch
    from rescan_line_sted_b200 import _lib, orientations, line_sted_tools as st

    base = st.psf_report('line', verbose=False, **bench.FIG2_2P0X_LR)['psfs']['rescan_sted']
    psfs = orientations.line_orientation_psfs(base, K, bench.EMISSION_2P0X_LR)
    brightness = bench.total_brightness(N)
    pinned_in = _lib.pinned_empty((1, N, N))
    pinned_in[...] = bench.synthetic_object(N)
    obj_t = torch.as_tensor(pinned_in).to('cuda:0', torch.float32)
    d = st.Deconvolver(psfs, output_prefix=os.path.join(tempfile.gettempdir(), 'lsted_dio_'),
                       verbose=False)

    def frame_numpy(seed):
        d.num_iterations = 0
        d.create_data_from_object(pinned_in, total_brightness=brightness, random_seed=seed)
        for _ in range(n_iter):
            d.iterate()
        return d.estimate

    def frame_tensor(seed):
        d.num_iterations = 0
        d.create_data_from_object(obj_t, total_brightness=brightness, random_seed=seed)
        for _ in range(n_iter):
            d.iterate()
        return d.tensor('estimate', torch.float32)

    def frame_resident(seed):
        h = d._handle
        h.set_option('forget_normalization', 1)
        h.simulate(brightness, seed)
        h.iterate(n_iter)

    def timed(fn, n):
        torch.cuda.synchronize()
        d._handle.sync()
        t0 = time.perf_counter()
        for s in range(n):
            fn(s + 1)
        torch.cuda.synchronize()
        d._handle.sync()
        return (time.perf_counter() - t0) * 1e3 / n

    x_np = pinned_in.copy()
    y_np = [pinned_in.copy() for _ in range(K)]
    y_t = [obj_t.clone() for _ in range(K)]
    ops = {'H numpy': lambda s: d.H(x_np), 'H tensor': lambda s: d.H(obj_t),
           'H_t numpy': lambda s: d.H_t(y_np), 'H_t tensor': lambda s: d.H_t(y_t)}
    frames = {'numpy': frame_numpy, 'tensor': frame_tensor, 'resident': frame_resident}
    for fn in list(frames.values()) + list(ops.values()):      # warm every shape
        fn(1000)
    ms = {k: [] for k in list(frames) + list(ops)}
    for _ in range(args.rounds):
        for name, fn in frames.items():
            ms[name].append(timed(fn, args.steps))
        for name, fn in ops.items():
            ms[name].append(timed(fn, args.steps))
    a = np.asarray(frame_numpy(5), dtype=np.float64)
    b = frame_tensor(5).double().cpu().numpy()
    out = {'card (name, power limit)': card(), 'size': N, 'orientations': K,
           'iterations': n_iter, 'steps': args.steps, 'rounds': args.rounds,
           'frames_per_s': {k: round(1000.0 / float(np.median(ms[k])), 2) for k in frames},
           'ms_per_frame_all_rounds': {k: [round(v, 2) for v in ms[k]] for k in frames},
           'ms_per_call': {k: round(float(np.median(ms[k])), 3) for k in ops},
           'estimate_rel_l2_numpy_vs_tensor_arm': float(np.linalg.norm(a - b) / np.linalg.norm(a))}
    print(json.dumps(out))


if __name__ == '__main__':
    main()
