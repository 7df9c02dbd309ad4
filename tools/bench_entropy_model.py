"""Deep-factorized entropy model on the GPU (DESIGN 3.10), in one process:

  (a) fused vs composed: fpcc_factorized_bits / _grad against the same definition composed in torch (fp32 autograd),
      timed window by window in alternation, at the latent of config 5's batch (4 x 200 k points, stride 2, L = 8) and
      at 1 M x 128.  GB/s over the algorithmic bytes (read y, params, dbits; write bits, dy, dparams), from shapes.
  (b) train_step_color step time at the config-5 shape in bf16, and the entropy model's share from a separate
      torch.profiler run.
  (c) the same step under DistributedDataParallel (one process per GPU, NCCL) at every world size out of 1 / 2 / 4 / 8
      the machine offers, global batch 8 split as 8 // world clouds per rank: weak-scaling samples/s.

usage: python tools/bench_entropy_model.py --out FILE [--windows 8] [--steps 10]
"""
import argparse
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


def composed_bits(y, params, bound=1e-9):
    """the definition of csrc/entropy_model.cu composed in torch ops (fp32, autograd; LowerBound as clamp with the
    straight gradient of compressai's rule left out: both paths are timed on inputs inside the bound)"""
    C = params.shape[0]
    sp = torch.nn.functional.softplus
    o, v_u, v_l = 0, (y + 0.5)[..., None], (y - 0.5)[..., None]
    for i, (r, c) in enumerate([(3, 1), (3, 3), (3, 3), (1, 3)]):
        H = sp(params[:, o:o + r * c].reshape(C, r, c)); o += r * c
        b = params[:, o:o + r]; o += r
        a = None
        if i < 3:
            a = torch.tanh(params[:, o:o + r]); o += r
        v_u = torch.einsum('coi,nci->nco', H, v_u) + b
        v_l = torch.einsum('coi,nci->nco', H, v_l) + b
        if a is not None:
            v_u = v_u + a * torch.tanh(v_u)
            v_l = v_l + a * torch.tanh(v_l)
    u, l = v_u[..., 0], v_l[..., 0]
    s = torch.where(u + l > 0, -1.0, 1.0)
    L = (torch.sigmoid(s * u) - torch.sigmoid(s * l)).abs()
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


def part_a(lines, windows):
    from fastpcc_b200 import ops
    from fastpcc_b200.entropy_models import NoisyDeepFactorizedEntropyModel
    shapes = [('config-5 latent', cfg5_latent_rows(), 8), ('1M x 128', 1000000, 128)]
    for name, n, C in shapes:
        torch.manual_seed(0)
        params = NoisyDeepFactorizedEntropyModel(C).params().detach().cuda()
        y = 3 * torch.randn((n, C), device='cuda')
        dbits = torch.rand((n, C), device='cuda')
        p_req = params.clone().requires_grad_()
        y_req = y.clone().requires_grad_()

        def fused_fwd():
            ops.factorized_bits(y, params)

        def fused_bwd():
            ops.factorized_grad(y, params, dbits)

        def comp_fwd():
            with torch.no_grad():
                composed_bits(y, params)

        def comp_bwd():
            torch.autograd.grad((composed_bits(y_req, p_req) * dbits).sum(), (y_req, p_req))

        # outputs agree (same definition; fp32 both)
        ref = composed_bits(y, params)
        diff = float(((ops.factorized_bits(y, params) - ref).abs() / ref.abs().clamp(min=1e-3)).max())
        iters = 20 if n * C < 1e7 else 5
        for f in (fused_fwd, fused_bwd, comp_fwd, comp_bwd):
            _time(f, 2)
        t = {k: [] for k in ('fused_fwd', 'fused_bwd', 'comp_fwd', 'comp_bwd')}
        for _ in range(windows):  # alternate window by window
            for k, f in (('fused_fwd', fused_fwd), ('comp_fwd', comp_fwd), ('fused_bwd', fused_bwd), ('comp_bwd', comp_bwd)):
                t[k].append(_time(f, iters))
        fwd_bytes = 4.0 * n * C * 2 + 4.0 * C * 43                      # read y, params; write bits
        bwd_bytes = 4.0 * n * C * 3 + 4.0 * C * 43 * 2                  # read y, dbits, params; write dy, dparams
        lines.append(f'(a) {name}: n = {n}, C = {C}, {n * C} elements; max rel diff fused vs composed bits {diff:.2e}')
        for k, nb in (('fused_fwd', fwd_bytes), ('comp_fwd', fwd_bytes), ('fused_bwd', bwd_bytes), ('comp_bwd', bwd_bytes)):
            med = float(np.median(t[k]))
            lines.append(f'    {k:10s} median {med:10.1f} us  (min {min(t[k]):.1f}, max {max(t[k]):.1f}, {windows} windows x {iters})'
                         f'  {nb / med / 1e3:8.1f} GB/s = {nb / med / 1e-6 / PEAK_BW:6.2%} of 7.7 TB/s')
        lines.append(f'    speed-up fused / composed: forward {np.median(t["comp_fwd"]) / np.median(t["fused_fwd"]):.1f}x, '
                     f'backward (fwd + grad) {np.median(t["comp_bwd"]) / np.median(t["fused_bwd"]):.1f}x')
        del y, dbits, y_req, p_req
        torch.cuda.empty_cache()


def _cfg5_batch(rank, per_rank, device):
    from fastpcc_b200 import synth, train
    clouds = [synth.colored_surface(900 + rank * per_rank + b, bits=10, n_target=CFG5_POINTS) for b in range(per_rank)]
    return train.make_color_batch([c[0] for c in clouds], [c[1] for c in clouds], device)


def part_b(lines, steps):
    from fastpcc_b200 import me as ME, train
    ME.set_compute_dtype(torch.bfloat16)
    torch.manual_seed(0)
    model = train.LossyColorNet(64).cuda()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    batch = _cfg5_batch(0, CFG5_CLOUDS, 'cuda')
    for _ in range(3):
        train.train_step_color(model, opt, batch)
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        train.train_step_color(model, opt, batch)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    lines.append(f'(b) train_step_color, LossyColorNet(64, L = 8), bf16, {CFG5_CLOUDS} x {CFG5_POINTS} points ({batch[0].shape[0]} rows): '
                 f'median {np.median(ts) * 1e3:.1f} ms / step (min {min(ts) * 1e3:.1f}, max {max(ts) * 1e3:.1f}, {steps} steps)')
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            train.train_step_color(model, opt, batch)
        torch.cuda.synchronize()
    tot, em = 0.0, 0.0
    for ev in prof.key_averages():
        dt = ev.device_time_total if hasattr(ev, 'device_time_total') else ev.cuda_time_total
        tot += dt
        if 'factorized' in ev.key:
            em += dt
            lines.append(f'    kernel {ev.key[:60]:60s} {dt / 3:9.1f} us / step')
    lines.append(f'    entropy-model kernels: {em / 3:.1f} us of {tot / 3:.1f} us device time per step = {em / max(tot, 1e-9):.3%} (profiler run)')
    ME.set_compute_dtype(torch.float16)


def _ddp_worker(rank, world, steps, q):
    import torch.distributed as dist
    from fastpcc_b200 import me as ME, train
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT='29659', RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', device_id=dev)
    ME.set_compute_dtype(torch.bfloat16)
    torch.manual_seed(0)
    ddp = torch.nn.parallel.DistributedDataParallel(train.LossyColorNet(64).to(dev), device_ids=[rank])
    opt = torch.optim.Adam(ddp.parameters(), lr=1e-3)
    per = 8 // world
    batch = _cfg5_batch(rank, per, dev)
    for _ in range(2):
        train.train_step_color(ddp, opt, batch)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        train.train_step_color(ddp, opt, batch)
    torch.cuda.synchronize()
    dist.barrier()
    dt = time.perf_counter() - t0
    if rank == 0:
        q.put(dt / steps)
    dist.destroy_process_group()


def part_c(lines, steps):
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    sizes = [w for w in (1, 2, 4, 8) if w <= n]
    ctx = mp.get_context('spawn')
    for w in sizes:
        q = ctx.Queue()
        procs = [ctx.Process(target=_ddp_worker, args=(r, w, steps, q)) for r in range(w)]
        for p in procs:
            p.start()
        step = q.get(timeout=900)
        for p in procs:
            p.join(timeout=120)
        lines.append(f'(c) DDP world {w}: {8 // w} clouds of {CFG5_POINTS} points per rank, {step * 1e3:.1f} ms / step, '
                     f'{8 / step:.1f} samples/s (global batch 8)')
    missing = [w for w in (1, 2, 4, 8) if w > n]
    if missing:
        lines.append(f'(c) world sizes {missing}: not measured (the machine has {n} GPU(s))')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--windows', type=int, default=8)
    ap.add_argument('--steps', type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_entropy_model: needs a GPU')
    lines = [f'card: {_card()}', f'torch {torch.__version__}, CUDA {torch.version.cuda}', '']
    part_a(lines, args.windows)
    lines.append('')
    part_b(lines, args.steps)
    lines.append('')
    part_c(lines, args.steps)
    text = '\n'.join(lines) + '\n'
    print(text)
    os.makedirs(osp.dirname(osp.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text)


if __name__ == '__main__':
    main()
