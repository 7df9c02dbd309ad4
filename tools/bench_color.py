"""Timing of the colour attributes on the device, in one process: the all-ties search fpcc_nn_tie_attr
(attributes.nearest_tie_attr) against the K = 1 search it extends (knn3d.knn_voxels) on the same clouds, alternated
window by window; attributes.recolor one- and two-way; metrics.pc_error with and without colours.

Clouds: an 800 k-point colour surface (synth.colored_surface) and its jittered copy (about 634 k points), and a LiDAR
frame with one constant colour.  CUDA events around `--iters` back-to-back calls after `--warmup` calls of the same
shape; every call includes its grid build and its workspace / output allocation.  Card name and power limit are read
in the same run.

    python tools/bench_color.py [--out profiles/r04_color.txt]
"""
import argparse
import os
import os.path as osp
import sys

import numpy as np
import torch

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))

from fastpcc_b200 import attributes, knn3d, metrics, synth  # noqa: E402
from tools.bench_knn import _card, _jittered, _time  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=osp.join('profiles', 'r04_color.txt'))
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--windows', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_color: no CUDA device')
    lines = []

    def say(s=''):
        print(s, flush=True)
        lines.append(s)

    say(f'device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, clocks.max.sm: {_card()}')
    say(f'torch {torch.__version__}, CUDA {torch.version.cuda}; warmup {args.warmup}, iters {args.iters}, '
        f'{args.windows} alternated windows per pair (ms per call, median of the windows)')
    surf, surf_rgb = synth.colored_surface(2, bits=11, n_target=800000)
    lidar = synth.lidar_frame(1)
    clouds = [('surface800k', surf, surf_rgb, _jittered(surf, 4)),
              ('lidar', lidar, np.full((lidar.shape[0], 3), 128, np.uint8), _jittered(lidar, 3))]
    say()
    say('search: queries = the jittered copy, reference = the cloud, (batch, x, y, z) rows')
    say(f'{"cloud":<14}{"nq":>9}{"nr":>9}{"knn_voxels K=1":>16}{"nearest_tie_attr":>18}{"ratio":>7}'
        f'{"mean ties":>11}{"max ties":>10}  d2 equal')
    for name, ref, rgb, qry in clouds:
        r, q = torch.from_numpy(synth.with_batch(ref)).cuda(), torch.from_numpy(synth.with_batch(qry)).cuda()
        c = torch.from_numpy(rgb).cuda()
        d1, _ = knn3d.knn_voxels(q, r, 1, n_batch=1)
        d2, n, _ = attributes.nearest_tie_attr(q, r, c, n_batch=1)
        same = torch.equal(d1.view(-1), d2)
        tk, tt = [], []
        for _ in range(args.windows):
            tk.append(_time(lambda: knn3d.knn_voxels(q, r, 1, n_batch=1), args.warmup, args.iters))
            tt.append(_time(lambda: attributes.nearest_tie_attr(q, r, c, n_batch=1), args.warmup, args.iters))
        mk, mt = float(np.median(tk)), float(np.median(tt))
        say(f'{name:<14}{qry.shape[0]:>9}{ref.shape[0]:>9}{mk:>16.3f}{mt:>18.3f}{mt / mk:>7.2f}'
            f'{n.double().mean().item():>11.3f}{int(n.max().item()):>10}  {same}')
        say(f'  windows: knn_voxels {", ".join(f"{t:.3f}" for t in tk)}; nearest_tie_attr '
            + ', '.join(f'{t:.3f}' for t in tt))

    org, org_rgb = torch.from_numpy(surf).cuda(), torch.from_numpy(surf_rgb).cuda()
    rec = torch.from_numpy(clouds[0][3]).cuda()
    say()
    say(f'recolor: {org.shape[0]} original points -> {rec.shape[0]} reconstructed points, (x, y, z) rows')
    for two_way in (False, True):
        ms = _time(lambda: attributes.recolor(org, org_rgb, rec, two_way=two_way), args.warmup, args.iters)
        say(f'  two_way={two_way!s:<6} {ms:8.3f} ms per call')

    rec_rgb = attributes.recolor(org, org_rgb, rec)
    say()
    say(f'pc_error: org {org.shape[0]} points, rec {rec.shape[0]} points (both directions, Hausdorff off), '
        'alternated windows of 5 calls')
    plain = metrics.pc_error(org, rec, 2048)
    col = metrics.pc_error(org, rec, 2048, org_colors=org_rgb, rec_colors=rec_rgb)
    say(f'  geometry keys identical with colours: {all(col[k] == v for k, v in plain.items())}; '
        f'c[0],PSNRF = {col["c[0],PSNRF"]:.4f}, c[1],PSNRF = {col["c[1],PSNRF"]:.4f}, '
        f'c[2],PSNRF = {col["c[2],PSNRF"]:.4f} dB (rec colours from recolor, two-way)')
    tp, tc = [], []
    for _ in range(args.windows):
        tp.append(_time(lambda: metrics.pc_error(org, rec, 2048), 1, 5))
        tc.append(_time(lambda: metrics.pc_error(org, rec, 2048, org_colors=org_rgb, rec_colors=rec_rgb), 1, 5))
    say('  geometry only:      ' + ', '.join(f'{t:.3f}' for t in tp) + ' ms per call')
    say('  geometry + colour:  ' + ', '.join(f'{t:.3f}' for t in tc) + ' ms per call')

    # kernel list of one nearest_tie_attr call (separate, profiled run)
    from torch.profiler import ProfilerActivity, profile
    r, q = torch.from_numpy(synth.with_batch(surf)).cuda(), torch.from_numpy(synth.with_batch(clouds[0][3])).cuda()
    attributes.nearest_tie_attr(q, r, org_rgb, n_batch=1)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        attributes.nearest_tie_attr(q, r, org_rgb, n_batch=1)
        knn3d.knn_voxels(q, r, 1, n_batch=1)
        torch.cuda.synchronize()
    say()
    say('kernels of one nearest_tie_attr call and one knn_voxels K = 1 call, surface800k (torch.profiler, profiled run; '
        'times include tracing):')
    evs = sorted(prof.key_averages(), key=lambda e: -e.device_time_total)
    for e in evs:
        if e.device_time_total > 0:
            say(f'  {e.device_time_total / 1e3:9.3f} ms  {e.count:3d}x  {e.key[:110]}')
    os.makedirs(osp.dirname(osp.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
