"""Timing of the point normals on the device, in one process: attributes.estimate_normals (fpcc_knn_normals: K-NN
walk, all-ties moment walk and 3 x 3 eigen solve fused in one kernel) at K in {8, 16, 32}, against
  - knn3d.knn_voxels at the same K on the same rows (the search alone: what the second walk and the solve add), and
  - a torch two-pass baseline: knn_voxels -> gather of the K neighbours -> moments in double -> torch.linalg.eigh
    (no ties past K, so not the same definition; the share of rows where both agree within 1e-3 is printed),
alternated window by window.  Clouds: an 800 k-point surface (synth.surface_cloud, 11 bits) and a LiDAR frame
(synth.lidar_frame, 16 bits).  CUDA events around `--iters` back-to-back calls after `--warmup` calls of the same
shape; every call includes its grid build and its workspace / output allocation.  Card name and power limit are read
in the same run; a kernel list of one call per variant comes from a separate, profiled run.

    python tools/bench_normals.py [--out profiles/r05_normals.txt]
"""
import argparse
import os
import os.path as osp
import sys

import numpy as np
import torch

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))

from fastpcc_b200 import attributes, knn3d, synth  # noqa: E402
from tools.bench_knn import _card, _time  # noqa: E402


def torch_two_pass(pts, K):
    """K nearest rows (lowest row on a tie) -> double moments -> batched eigh -> least eigenvector, largest |c| > 0"""
    _, idx = knn3d.knn_voxels(pts, pts, K)
    x = pts.double()
    d = x[idx.long()] - x[:, None, :]                       # [n, K, 3]
    s = d.sum(1)
    m = K * torch.einsum('nki,nkj->nij', d, d) - s[:, :, None] * s[:, None, :]
    # cuSOLVER's batched solver rejected one batch of 800 k matrices (CUSOLVER_STATUS_INVALID_VALUE): chunks of 32 k
    v = torch.cat([torch.linalg.eigh(c)[1][:, :, 0] for c in m.split(1 << 15)])
    top = v.gather(1, v.abs().argmax(1, keepdim=True))
    return torch.where(top < 0, -v, v).float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=osp.join('profiles', 'r05_normals.txt'))
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--windows', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_normals: no CUDA device')
    lines = []

    def say(s=''):
        print(s, flush=True)
        lines.append(s)

    say(f'device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, clocks.max.sm: {_card()}')
    say(f'torch {torch.__version__}, CUDA {torch.version.cuda}; warmup {args.warmup}, iters {args.iters}, '
        f'{args.windows} alternated windows per variant (ms per call, median of the windows)')
    clouds = [('surface800k', synth.surface_cloud(2, bits=11, n_target=800000)), ('lidar', synth.lidar_frame(1))]
    say()
    say('one cloud per call, (x, y, z) rows; queries = references = the cloud')
    say(f'{"cloud":<13}{"n":>8}{"K":>4}{"knn_voxels":>12}{"estimate_normals":>18}{"torch 2-pass":>14}'
        f'{"normals/knn":>13}{"2-pass/normals":>16}{"zero rows":>11}{"agree":>8}')
    for name, xyz in clouds:
        pts = torch.from_numpy(xyz).cuda()
        for K in (8, 16, 32):
            nrm = attributes.estimate_normals(pts, K)
            base = torch_two_pass(pts, K)
            zero = (nrm == 0).all(1)
            agree = (torch.minimum((nrm - base).abs().amax(1), (nrm + base).abs().amax(1)) < 1e-3)[~zero]
            tk, tn, tb = [], [], []
            for _ in range(args.windows):
                tk.append(_time(lambda: knn3d.knn_voxels(pts, pts, K), args.warmup, args.iters))
                tn.append(_time(lambda: attributes.estimate_normals(pts, K), args.warmup, args.iters))
                tb.append(_time(lambda: torch_two_pass(pts, K), args.warmup, args.iters))
            mk, mn, mb = (float(np.median(t)) for t in (tk, tn, tb))
            say(f'{name:<13}{xyz.shape[0]:>8}{K:>4}{mk:>12.3f}{mn:>18.3f}{mb:>14.3f}{mn / mk:>13.2f}{mb / mn:>16.2f}'
                f'{zero.double().mean().item():>11.4f}{agree.double().mean().item():>8.4f}')
            say('  windows: knn_voxels ' + ', '.join(f'{t:.3f}' for t in tk) + '; estimate_normals '
                + ', '.join(f'{t:.3f}' for t in tn) + '; torch 2-pass ' + ', '.join(f'{t:.3f}' for t in tb))

    from torch.profiler import ProfilerActivity, profile
    pts = torch.from_numpy(clouds[0][1]).cuda()
    attributes.estimate_normals(pts, 16)
    torch_two_pass(pts, 16)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        attributes.estimate_normals(pts, 16)
        knn3d.knn_voxels(pts, pts, 16)
        torch_two_pass(pts, 16)
        torch.cuda.synchronize()
    say()
    say('kernels of one estimate_normals, one knn_voxels and one torch 2-pass call at K = 16, surface800k '
        '(torch.profiler, profiled run; times include tracing):')
    for e in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
        if e.device_time_total > 0:
            say(f'  {e.device_time_total / 1e3:9.3f} ms  {e.count:3d}x  {e.key[:110]}')
    os.makedirs(osp.dirname(osp.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
