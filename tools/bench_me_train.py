"""Training step of the lossy geometry net on the MinkowskiEngine shim: forward + backward + Adam step of
`train.LossyGeoNet`, on the tcgen05 forward / dgrad / wgrad kernels with `fpcc_kmap_transpose` and `fpcc_act_grad_f16`,
against the same net on a torch autograd path (per-offset index_select + matmul + index_add, same compute dtype),
alternated window by window in one process.
usage: python tools/bench_me_train.py [--steps 5] [--windows 3] [--out profiles/r06_me_train.txt]

Workloads: one 800 k-point surface cloud (config 4's working shape) and a batch of 4 x 200 k partitions (config 5's),
in bf16 and in fp16 (with a GradScaler).  Then, per workload, an instrumented pass (CUDA events around every C-ABI call,
algorithmic ops / bytes from shapes): dgrad TFLOP/s (spconv calls of the full step minus those of the forward alone),
wgrad TFLOP/s (2 P C_in C_out), and the GB/s of act_grad_f16 / kmap_transpose against 7.7 TB/s.  Last, a torch.profiler
run of two steps lists the CUDA kernels by time."""
import argparse
import io
import json
import os.path as osp
import subprocess
import sys
import time

import torch

sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))
from fastpcc_b200 import autograd, me as ME, ops, synth, train  # noqa: E402

HBM_TBS = 7.7  # B200 data sheet, one GPU


def torch_me_layer(feats, kernel, bias, spec, run):
    """baseline: the layer's forward written with torch ops (autograd differentiates it); same kernel map and dtype"""
    dt = spec.dtype
    w = _kio_grad(kernel, spec.layout).to(dt)
    f = feats.to(dt)
    if spec.kind in ('conv', 'tconv'):
        in_map, out_map, off = autograd._compacted(spec.table, f.shape[0])
        out = torch.zeros((spec.table.shape[1], spec.c_out), dtype=dt, device=f.device)
        for k in range(len(off) - 1):
            s, e = off[k], off[k + 1]
            if e > s:
                out = out.index_add(0, out_map[s:e].long(), torch.index_select(f, 0, in_map[s:e].long()) @ w[k])
    elif spec.kind == 'linear':
        out = f @ w[0]
    else:
        out = (f @ w.permute(1, 0, 2).reshape(spec.c_in, -1)).reshape(-1, spec.c_out)
    if bias is not None:
        out = out + bias.reshape(1, -1).to(dt)
    if spec.act == ops.ACT_RELU:
        out = torch.relu(out)
    elif spec.act == ops.ACT_LEAKY:
        out = torch.nn.functional.leaky_relu(out, spec.slope)
    return out.float() if spec.c_out == 1 else out


def _kio_grad(kernel, layout):
    return kernel if layout == 'kio' else (kernel[None] if layout == 'io' else kernel.t()[None])


def workloads():
    one = train.make_lossy_batch([synth.surface_cloud(41, bits=10, n_target=800000)], 'cuda')
    four = train.make_lossy_batch([synth.surface_cloud(50 + i, bits=10, n_target=200000) for i in range(4)], 'cuda')
    return {'800k x1': one, '200k x4': four}


def make(dt):
    ME.set_compute_dtype(dt)
    torch.manual_seed(0)
    model = train.LossyGeoNet(64).cuda()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler('cuda') if dt == torch.float16 else None
    return model, opt, scaler


def timed(model, opt, scaler, batch, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = train.train_step_lossy(model, opt, batch, scaler)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps, float(loss)


def instrumented(model, opt, scaler, batch):
    prof = ops.enable_profile(True)
    with torch.enable_grad():
        model(batch)
    fwd = ops.profile_summary(prof)
    prof = ops.enable_profile(True)
    train.train_step_lossy(model, opt, batch, scaler)
    full = ops.profile_summary(prof)
    ops.enable_profile(False)
    row = {}
    f, b = fwd.get('spconv_f16_tc', {}), full.get('spconv_f16_tc', {})
    if b:
        ms, fl = b['ms'] - f.get('ms', 0.0), b['ops'] - f.get('ops', 0.0)
        row['dgrad_spconv'] = {'ms': round(ms, 3), 'tflops': round(fl / (ms * 1e-3) / 1e12, 1) if ms > 0 else None}
    for tag, key in (('spconv_wgrad_tc', 'wgrad'),):
        if tag in full:
            v = full[tag]
            row[key] = {'ms': round(v['ms'], 3), 'tflops': round(v['ops'] / (v['ms'] * 1e-3) / 1e12, 1), 'launches': v['launches']}
    for tag in ('fpcc_act_grad_f16', 'fpcc_kmap_transpose'):
        if tag in full:
            v = full[tag]
            gbs = v['bytes'] / (v['ms'] * 1e-3) / 1e9
            row[tag] = {'ms': round(v['ms'], 3), 'GB/s': round(gbs, 1), 'share_of_hbm': round(gbs / (HBM_TBS * 1e3), 3),
                        'bound': 'memory (HBM bytes)', 'launches': v['launches']}
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--windows', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    out = io.StringIO()
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    print(f'# {torch.cuda.get_device_name()} | nvidia-smi: {smi}', file=out)
    print(f'# steps per window {args.steps}, windows {args.windows}, warm-up {args.warmup} steps per (workload, dtype, path)', file=out)
    data = workloads()
    kernel_layer = autograd.me_layer
    for name, batch in data.items():
        for dt in (torch.bfloat16, torch.float16):
            res = {'kernels': [], 'torch': []}
            models = {p: make(dt) for p in res}
            for p in res:
                autograd.me_layer = kernel_layer if p == 'kernels' else torch_me_layer
                timed(*models[p], batch, args.warmup)
            for _ in range(args.windows):
                for p in res:
                    autograd.me_layer = kernel_layer if p == 'kernels' else torch_me_layer
                    res[p].append(timed(*models[p], batch, args.steps))
            autograd.me_layer = kernel_layer
            ms = {p: sorted(x[0] for x in v)[len(v) // 2] for p, v in res.items()}
            row = {'workload': name, 'points': int(batch.shape[0]), 'dtype': str(dt).split('.')[-1],
                   'ms_per_step_median': {p: round(v, 2) for p, v in ms.items()},
                   'ms_per_step_windows': {p: [round(x[0], 2) for x in v] for p, v in res.items()},
                   'speedup': round(ms['torch'] / ms['kernels'], 2),
                   'loss_last': {p: round(v[-1][1], 4) for p, v in res.items()},
                   'instrumented': instrumented(*models['kernels'], batch)}
            print(json.dumps(row), file=out)
            print(json.dumps(row), flush=True)
            del models
            torch.cuda.empty_cache()
    # kernel table of a separate profiler run (bf16, the single 800 k cloud)
    model, opt, scaler = make(torch.bfloat16)
    batch = data['800k x1']
    train.train_step_lossy(model, opt, batch, scaler)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):
            train.train_step_lossy(model, opt, batch, scaler)
        torch.cuda.synchronize()
    print('# torch.profiler, bf16, 800k x1, 2 steps: CUDA kernels by total time', file=out)
    try:
        table = prof.key_averages().table(sort_by='self_device_time_total', row_limit=25, max_name_column_width=70)
    except (AttributeError, KeyError, ValueError):
        table = prof.key_averages().table(sort_by='self_cuda_time_total', row_limit=25, max_name_column_width=70)
    print(table, file=out)
    text = out.getvalue()
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text)
    print(text)


if __name__ == '__main__':
    main()
