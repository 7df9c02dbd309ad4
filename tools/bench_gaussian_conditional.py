"""Gaussian conditional entropy model and mean-scale hyperprior on the GPU (DESIGN 3.11), in one process:

  (a) fused vs composed: fpcc_gaussian_bits / _grad against the same definition composed in torch (fp32, forward +
      autograd backward), timed window by window in alternation, at the config-5 latent (4 x 200 k points, stride 2,
      L = 8) and at 1 M x 128 (larger than L2).  GB/s over the algorithmic bytes, from shapes.
  (b) update(): the device tables of the default scale table (fpcc_gaussian_pmf + fpcc_pmf_to_quantized_cdf).
  (c) compress / decompress of the config-5 latent (one indexed stream; the decoder is one warp's serial chain).
  (d) train_step_color at 4 x 200 k points in bf16, prior='hyperprior' against 'factorized' alternated, and the
      entropy models' share of device time from a separate torch.profiler run.

usage: python tools/bench_gaussian_conditional.py --out FILE [--windows 8] [--steps 10]
"""
import argparse
import math
import os
import os.path as osp
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))

PEAK_BW = 7.7e12  # B/s, HGX B200 data sheet, one GPU
CFG5_POINTS, CFG5_CLOUDS = 200000, 4


def _card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def composed_bits(y, scales, means, scale_bound=0.11, bound=1e-9):
    """the definition of csrc/entropy_model.cu composed in torch ops (fp32, autograd; the bounds as clamps: both paths
    are timed on the same inputs and the lower-bound gradient rule is left out of the composed one)"""
    v = (y - means).abs()
    s = scales.clamp(min=scale_bound)
    c = lambda x: 0.5 * torch.special.erfc(-x * (0.5 ** 0.5))  # noqa: E731
    L = c((0.5 - v) / s) - c((-0.5 - v) / s)
    return -torch.log2(L.clamp(min=bound))


def cfg5_latent_rows():
    from fastpcc_b200 import synth
    n = 0
    for b in range(CFG5_CLOUDS):
        xyz, _ = synth.colored_surface(500 + b, bits=10, n_target=CFG5_POINTS)
        n += np.unique(xyz >> 1, axis=0).shape[0]
    return n


def _time(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters  # us per call


def _inputs(n, C, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    ms = torch.empty((n, 2 * C), device='cuda')
    ms[:, :C] = 10 * torch.randn((n, C), device='cuda', generator=g)
    ms[:, C:] = torch.exp(torch.empty((n, C), device='cuda').uniform_(math.log(0.05), math.log(50.0), generator=g))
    mu, sigma = ms[:, :C], ms[:, C:]                                   # column halves, as h_s writes them
    y = mu + sigma * torch.randn((n, C), device='cuda', generator=g)
    return y, mu, sigma


def part_a(lines, windows):
    from fastpcc_b200 import ops
    for name, n, C in [('config-5 latent', cfg5_latent_rows(), 8), ('1M x 128', 1000000, 128)]:
        y, mu, sigma = _inputs(n, C)
        dbits = torch.rand((n, C), device='cuda')
        y_r, m_r, s_r = (t.clone().requires_grad_() for t in (y, mu, sigma))

        def fused_fwd():
            ops.gaussian_bits(y, sigma, mu)

        def fused_bwd():
            ops.gaussian_grad(y, sigma, dbits, mu)

        def comp_fwd():
            with torch.no_grad():
                composed_bits(y, sigma, mu)

        def comp_bwd():
            torch.autograd.grad((composed_bits(y_r, s_r, m_r) * dbits).sum(), (y_r, s_r, m_r))

        ref = composed_bits(y, sigma, mu)
        diff = float(((ops.gaussian_bits(y, sigma, mu) - ref).abs() / ref.abs().clamp(min=1e-3)).max())
        iters = 50 if n * C < 1e7 else 10
        for f in (fused_fwd, fused_bwd, comp_fwd, comp_bwd):
            _time(f, 2)
        t = {k: [] for k in ('fused_fwd', 'fused_bwd', 'comp_fwd', 'comp_bwd')}
        for _ in range(windows):  # alternate window by window
            for k, f in (('fused_fwd', fused_fwd), ('comp_fwd', comp_fwd), ('fused_bwd', fused_bwd), ('comp_bwd', comp_bwd)):
                t[k].append(_time(f, iters))
        fwd_bytes = 4.0 * n * C * 4                                    # read y, mu, sigma; write bits
        bwd_bytes = 4.0 * n * C * 7                                    # read y, mu, sigma, dbits; write dy, dmu, dsigma
        lines.append(f'(a) {name}: n = {n}, C = {C}, {n * C} elements; max rel diff fused vs composed bits {diff:.2e}')
        for k, nb in (('fused_fwd', fwd_bytes), ('comp_fwd', fwd_bytes), ('fused_bwd', bwd_bytes), ('comp_bwd', bwd_bytes)):
            med = float(np.median(t[k]))
            lines.append(f'    {k:10s} median {med:10.1f} us  (min {min(t[k]):.1f}, max {max(t[k]):.1f}, {windows} windows x {iters})'
                         f'  {nb / med / 1e3:8.1f} GB/s = {nb / med / 1e-6 / PEAK_BW:6.2%} of 7.7 TB/s')
        lines.append(f'    speed-up fused / composed: forward {np.median(t["comp_fwd"]) / np.median(t["fused_fwd"]):.1f}x, '
                     f'fwd + grad vs fwd + autograd bwd '
                     f'{np.median(t["comp_bwd"]) / (np.median(t["fused_fwd"]) + np.median(t["fused_bwd"])):.1f}x')
        del y, mu, sigma, dbits, y_r, m_r, s_r
        torch.cuda.empty_cache()


def part_bc(lines):
    from fastpcc_b200 import ops
    from fastpcc_b200.entropy_models import GaussianConditionalEntropyModel
    em = GaussianConditionalEntropyModel().cuda().eval()
    em.update()
    torch.cuda.synchronize()
    ts, tp = [], []
    for _ in range(5):
        t0 = time.perf_counter()
        em.update()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        pmf, offs = ops.gaussian_pmf(em.scale_table)
        torch.cuda.synchronize()
        tp.append(_time(lambda: ops.gaussian_pmf(em.scale_table), 5))
    lens = em._tables[2]
    from fastpcc_b200 import _lib
    from fastpcc_b200.ops import _p, _s
    T, S = pmf.shape
    cdf = torch.empty((T, S + 2), dtype=torch.int32, device='cuda')
    ln = torch.empty(T, dtype=torch.int32, device='cuda')
    tq = []
    for _ in range(5):
        p2, o2 = pmf.clone(), offs.clone()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.call('fpcc_pmf_to_quantized_cdf', _p(p2), T, S, _p(o2), 1, _p(cdf), _p(ln), _s())
        e1.record()
        torch.cuda.synchronize()
        tq.append(e0.elapsed_time(e1) * 1e3)
    lines.append(f'(b) update(), 64 scales, tail_mass 1e-9: pmf [64, {pmf.shape[1]}]; median {np.median(ts) * 1e3:.2f} ms '
                 f'(min {min(ts) * 1e3:.2f}; host clock to a synchronise, incl. the host read of the table) of which '
                 f'fpcc_gaussian_pmf {np.median(tp):.1f} us and fpcc_pmf_to_quantized_cdf (one thread per table) '
                 f'{np.median(tq):.1f} us (events); table lengths {int(lens.min())} .. {int(lens.max())}')
    n, C = cfg5_latent_rows(), 8
    y, mu, sigma = _inputs(n, C, 1)
    data = em.compress(y, sigma, mu)
    em.decompress(data, sigma, mu)
    tc, td = [], []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        data = em.compress(y, sigma, mu)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        y_hat = em.decompress(data, sigma, mu)
        torch.cuda.synchronize()
        tc.append(t1 - t0)
        td.append(time.perf_counter() - t1)
    ok = torch.equal(y_hat, torch.round(y - mu) + mu)
    lines.append(f'(c) config-5 latent {n} x {C}: {len(data)} bytes ({8 * len(data) / (n * C):.3f} bits per element), '
                 f'compress median {np.median(tc) * 1e3:.1f} ms, decompress median {np.median(td) * 1e3:.1f} ms '
                 f'(one stream: one warp decodes {n * C} symbols in series); round trip exact: {ok}')


def part_d(lines, steps):
    from fastpcc_b200 import me as ME, synth, train
    ME.set_compute_dtype(torch.bfloat16)
    clouds = [synth.colored_surface(900 + b, bits=10, n_target=CFG5_POINTS) for b in range(CFG5_CLOUDS)]
    batch = train.make_color_batch([c[0] for c in clouds], [c[1] for c in clouds], 'cuda')
    nets = {}
    for prior in ('factorized', 'hyperprior'):
        torch.manual_seed(0)
        model = train.LossyColorNet(64, prior=prior).cuda()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        for _ in range(3):
            train.train_step_color(model, opt, batch)
        nets[prior] = (model, opt)
    torch.cuda.synchronize()
    ts = {k: [] for k in nets}
    for _ in range(steps):                                             # alternated step by step
        for prior, (model, opt) in nets.items():
            t0 = time.perf_counter()
            train.train_step_color(model, opt, batch)
            torch.cuda.synchronize()
            ts[prior].append(time.perf_counter() - t0)
    for prior in nets:
        lines.append(f'(d) train_step_color, LossyColorNet(64, L = 8, prior={prior!r}), bf16, {CFG5_CLOUDS} x {CFG5_POINTS} '
                     f'points ({batch[0].shape[0]} rows): median {np.median(ts[prior]) * 1e3:.1f} ms / step '
                     f'(min {min(ts[prior]) * 1e3:.1f}, max {max(ts[prior]) * 1e3:.1f}, {steps} steps)')
    from torch.profiler import ProfilerActivity, profile
    model, opt = nets['hyperprior']
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            train.train_step_color(model, opt, batch)
        torch.cuda.synchronize()
    tot, em = 0.0, 0.0
    for ev in prof.key_averages():
        dt = ev.device_time_total if hasattr(ev, 'device_time_total') else ev.cuda_time_total
        tot += dt
        if 'gaussian' in ev.key or 'factorized' in ev.key:
            em += dt
            lines.append(f'    kernel {ev.key[:60]:60s} {dt / 3:9.1f} us / step')
    lines.append(f'    entropy-model kernels (Gaussian conditional + the hyper-latent\'s factorized prior): {em / 3:.1f} us of '
                 f'{tot / 3:.1f} us device time per step = {em / max(tot, 1e-9):.3%} (profiler run; h_a / h_s layers not counted)')
    ME.set_compute_dtype(torch.float16)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--windows', type=int, default=8)
    ap.add_argument('--steps', type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_gaussian_conditional: needs a GPU')
    lines = [f'card: {_card()}', f'torch {torch.__version__}, CUDA {torch.version.cuda}', '']
    part_a(lines, args.windows)
    lines.append('')
    part_bc(lines)
    lines.append('')
    part_d(lines, args.steps)
    text = '\n'.join(lines) + '\n'
    print(text)
    os.makedirs(osp.dirname(osp.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text)


if __name__ == '__main__':
    main()
