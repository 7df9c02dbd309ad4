"""Timing of the cell-grid K-NN (fpcc_knn_search) on the device, in one process: knn_voxels (int32) and knn_points
(float32) at K in {1, 8, 16, 32} on a LiDAR frame and an 800 k-point surface cloud, and metrics.pc_error at 800 k on
the grid path and on the brute-force fpcc_nn_search, alternated in the same run.

CUDA events around `--iters` back-to-back calls after `--warmup` calls of the same shape; every call includes its grid
build (bounding boxes, sort, cell table) and its workspace / output allocation.  HBM share: the least traffic a call
needs (reference rows read once, query rows read once, outputs written once, 16 B per row of coordinates, 12 B per
neighbour) over 7.7 TB/s, against the measured time.  Card name and power limit are read in the same run.

    python tools/bench_knn.py [--out profiles/r03_knn.txt]
"""
import argparse
import os
import os.path as osp
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))

from fastpcc_b200 import knn3d, metrics, synth  # noqa: E402

HBM_BPS = 7.7e12  # HGX B200 data sheet, one GPU


def _jittered(xyz, seed, keep=0.8):
    rng = np.random.default_rng(seed)
    out = xyz + rng.integers(-2, 3, xyz.shape)
    return np.unique(out.astype(np.int32)[rng.random(xyz.shape[0]) < keep], axis=0)


def _time(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def _card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else 'nvidia-smi gave no output'
    except (OSError, subprocess.SubprocessError) as e:
        return f'nvidia-smi unavailable ({e})'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=osp.join('profiles', 'r03_knn.txt'))
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--brute-reps', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_knn: no CUDA device')
    lines = []

    def say(s=''):
        print(s, flush=True)
        lines.append(s)

    say(f'device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, clocks.max.sm: {_card()}')
    say(f'torch {torch.__version__}, CUDA {torch.version.cuda}; warmup {args.warmup}, iters {args.iters}; '
        f'HBM bound at {HBM_BPS / 1e12:.1f} TB/s (data sheet)')
    lidar = synth.lidar_frame(1)
    surf = synth.surface_cloud(2, bits=11, n_target=800000)
    clouds = [('lidar', lidar, _jittered(lidar, 3)), ('surface800k', surf, _jittered(surf, 4))]
    say()
    say(f'{"what":<34}{"nq":>9}{"nr":>9}{"K":>4}{"ms/call":>10}{"Mq/s":>9}{"MB min":>9}{"HBM %":>7}')
    for name, ref, qry in clouds:
        for kind in ('knn_voxels', 'knn_points'):
            if kind == 'knn_voxels':
                r, q = torch.from_numpy(synth.with_batch(ref)).cuda(), torch.from_numpy(synth.with_batch(qry)).cuda()
            else:
                r = torch.from_numpy(ref.astype(np.float32)).cuda()[None]
                q = torch.from_numpy(qry.astype(np.float32)).cuda()[None]
            nq, nr = qry.shape[0], ref.shape[0]
            for k in (1, 8, 16, 32):
                if kind == 'knn_voxels':
                    fn = lambda: knn3d.knn_voxels(q, r, k, n_batch=1)  # noqa: E731
                else:
                    fn = lambda: knn3d.knn_points(q, r, K=k)  # noqa: E731
                ms = _time(fn, args.warmup, args.iters)
                byts = nr * 16 + nq * 16 + nq * k * 12
                share = byts / HBM_BPS / (ms * 1e-3) * 100
                say(f'{kind + " " + name:<34}{nq:>9}{nr:>9}{k:>4}{ms:>10.3f}{nq / ms / 1e3:>9.1f}{byts / 1e6:>9.1f}'
                    f'{share:>7.2f}')
    # pc_error at 800 k, both searches, alternated
    org, rec = torch.from_numpy(surf).cuda(), torch.from_numpy(clouds[1][2]).cuda()
    say()
    say(f'pc_error: org {org.shape[0]} points, rec {rec.shape[0]} points (both directions, Hausdorff on)')
    grid = metrics.pc_error(org, rec, 2048, hausdorff=True)
    brute = metrics.pc_error(org, rec, 2048, hausdorff=True, search=metrics.nn_search_bruteforce)
    say(f'  results identical on every key: {grid == brute}  (mseF,PSNR (p2point) = {grid["mseF,PSNR (p2point)"]:.6f})')
    tg, tb = [], []
    for _ in range(args.brute_reps):
        tg.append(_time(lambda: metrics.pc_error(org, rec, 2048, hausdorff=True), 1, 5))
        tb.append(_time(lambda: metrics.pc_error(org, rec, 2048, hausdorff=True,
                                                 search=metrics.nn_search_bruteforce), 0, 1))
    say(f'  grid (fpcc_knn_search, K = 1):  ms per pc_error call, {args.brute_reps} windows of 5: '
        + ', '.join(f'{t:.2f}' for t in tg))
    say(f'  brute force (fpcc_nn_search):   ms per pc_error call, {args.brute_reps} single calls:  '
        + ', '.join(f'{t:.1f}' for t in tb))
    say(f'  speed-up (median): {np.median(tb) / np.median(tg):.0f}x')
    # kernel list of one knn_voxels call (separate, profiled run)
    from torch.profiler import ProfilerActivity, profile
    r, q = torch.from_numpy(synth.with_batch(surf)).cuda(), torch.from_numpy(synth.with_batch(clouds[1][2])).cuda()
    knn3d.knn_voxels(q, r, 16, n_batch=1)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        knn3d.knn_voxels(q, r, 16, n_batch=1)
        torch.cuda.synchronize()
    say()
    say('kernels of one knn_voxels call, surface800k, K = 16 (torch.profiler, profiled run; times include tracing):')
    evs = sorted(prof.key_averages(), key=lambda e: -e.device_time_total)
    for e in evs:
        if e.device_time_total > 0:
            say(f'  {e.device_time_total / 1e3:9.3f} ms  {e.count:3d}x  {e.key[:110]}')
    os.makedirs(osp.dirname(osp.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
