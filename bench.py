#!/usr/bin/env python
"""bench.py -- encode+decode throughput of the lossless LiDAR geometry codec hot path on B200.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on
rank 0.  A "step" = compress + decompress of `--frames` synthetic KITTI-shaped scans (S2 "lidar-120k",
SURVEY.md 8d) per GPU through models/convolutional/lossl_coord_int's B200-native twin
(fastpcc_b200.lossl_coord_int.Model, default 256-channel config).  Frames are independent, so ranks share
nothing: weak scaling, no data-path collective; the only collectives are the barrier and the max-over-ranks
of the timed region.

  value     Mpts/s with the voxelised frames already resident in HBM (CUDA events, max over ranks)
  e2e       same metric through the public API from HOST buffers: H2D of the coordinates, D2H of the
            bitstream, H2D of the bitstream, D2H of the decoded coordinates, all inside the timed region
  roofline  the tcgen05 sparse-conv kernel: algorithmic int8 OPs (2*pairs*Cin*Cout) / its CUDA-event time
  cpu_baseline  the CPU oracle (numpy port of the reference path) on a bounded sample of the same workload

`--dump-outputs DIR` writes what the last timed step returned (the bitstream and the decoded coordinates of every frame
on rank 0; with `--impl reference`, of its sample) as DIR/<name>.npy, so that two builds of the project can be compared
output for output on identical inputs.

`--impl reference` times the reference path on the host cores: the oracle port of the codec on a multi-threaded
backend (torch-CPU SGEMM + OpenMP C kernels) with the reference's own compiled range coder (the reference's GPU
extension needs MinkowskiEngine/torchsparse/a CUTLASS fork, none installable offline).
"""
import argparse
import json
import os
import os.path as osp
import subprocess
import sys
import time

import numpy as np

ROOT = osp.dirname(osp.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(channels=256, max_stride_wo_recurrent=2048, max_stride=8192, fea_stride=16)
WORKLOAD = ('lossl_coord LiDAR lossless (BASELINE configs[1]: KITTI-shaped synthetic scans ~120k pts/frame, 16-bit grid, '
            'C=256 default topology) coded by its integer-only inference path lossl_coord_int (configs[2], bit-exact bitstreams)')


def load_peaks():
    p = osp.join(ROOT, 'MEASURED_PEAKS.json')
    if osp.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return d, 'measured'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


class ClockSampler:
    """One long-lived `nvidia-smi -lms` process logging clocks / throttle reasons of one GPU during the timed region
    (spawning nvidia-smi repeatedly from Python perturbs the run it is supposed to watch)."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '250'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            pass

    def start(self):
        pass

    def summary(self):
        samples = []
        if self.proc is not None:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
                samples = [[v.strip() for v in line.split(',')] for line in out.strip().splitlines() if line.count(',') >= 6]
            except Exception:
                self.proc.kill()
        if not samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(s[0]) for s in samples)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith('active') for s in samples)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(samples[0][1]), 'reasons': reasons,
                'samples': len(sm), 'power_w_max': max(float(s[2]) for s in samples)}


def make_frames(n, rank, world=1):
    """This rank's frames of the job: the job is `world * n` independent scans (unit u = scan of seed 1000 + u); the units
    are dealt to the ranks by fastpcc_b200.sharding (size-balanced assignment, no data-path collective) and every rank
    generates only its own."""
    from concurrent.futures import ThreadPoolExecutor
    from fastpcc_b200 import sharding, synth
    units = sharding.local_indices([1] * (world * n), rank=rank, world=world)
    workers = max(1, min(8, (os.cpu_count() or 1) // max(1, world)))  # numpy releases the GIL in the heavy parts
    with ThreadPoolExecutor(max_workers=workers) as pool:
        return list(pool.map(lambda u: synth.with_batch(synth.lidar_frame(1000 + u)), units))


def _sample_rows(n, cap, seed=0):
    """Sorted row indices of a fixed seeded sample of `cap` of `n` rows (all rows when n <= cap): the same n gives the
    same rows in every run."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))


def dump_outputs(out_dir, data, rec, max_bytes=1 << 22, max_rows=1 << 21):
    """Writes one step's result as float arrays (exact: bytes and 16-bit grid coordinates fit float32), 40 MB at most:

      bitstream_sizes.npy  float64 [frames]             bytes of every frame's bitstream
      bitstream_bytes.npy  float32 [<= max_bytes]       the concatenated bitstreams, or a seeded sample of their bytes
      decoded_sizes.npy    float64 [frames]             points of every decoded frame
      decoded_xyz.npy      float32 [<= max_rows, 3]     the concatenated decoded frames, or a seeded sample of their rows
    """
    import torch
    os.makedirs(out_dir, exist_ok=True)
    stream = np.frombuffer(b''.join(data), dtype=np.uint8)
    cat = torch.cat([torch.as_tensor(r) for r in rec])
    rows = torch.from_numpy(_sample_rows(cat.shape[0], max_rows)).to(cat.device)
    out = {
        'bitstream_sizes': np.array([len(d) for d in data], dtype=np.float64),
        'bitstream_bytes': stream[_sample_rows(stream.size, max_bytes)].astype(np.float32),
        'decoded_sizes': np.array([r.shape[0] for r in rec], dtype=np.float64),
        'decoded_xyz': cat.index_select(0, rows).cpu().numpy().astype(np.float32),
    }
    for name, a in out.items():
        np.save(osp.join(out_dir, name + '.npy'), a)
    sys.stderr.write(f'[bench] outputs of the last timed step: {", ".join(f"{k} {v.shape}" for k, v in out.items())} -> {out_dir}\n')


def cpu_arm_model(cores):
    """The reference path on the host cores: oracle/lossl_coord_int.py (the codec's control flow, pinned to the reference
    Python by tests/golden) on the multi-threaded backend oracle/int_ops_fast.py (torch-CPU SGEMM for the per-offset
    GEMMs of cuda_ops.py:153-166, OpenMP C for the element-wise epilogues and the CDF head) with the REFERENCE'S OWN
    compiled range coder (oracle/_ref, built from /root/reference) when it is present, else the C restatement."""
    import ctypes
    import torch
    from fastpcc_b200 import synth
    from oracle import build_ref, int_ops_fast, lossl_coord_int as M
    torch.set_num_threads(cores)
    try:  # torchrun exports OMP_NUM_THREADS=1: the OpenMP kernels of the arm must still use every core
        ctypes.CDLL('libgomp.so.1').omp_set_num_threads(cores)
    except OSError:
        pass
    M.K = int_ops_fast
    ref = build_ref.load_ref('simple_rans_ext_cpp')
    coder = 'range coder: C restatement (oracle/rans_oracle.c)'
    if ref is not None:
        M.RansEncoder, M.RansDecoder = ref.RansEncoder, ref.RansDecoder
        coder = "range coder: the reference's own compiled C++ (oracle/_ref)"
    sd = synth.make_lossl_int_state_dict(seed=7, **CFG)
    return M.Model(sd, **CFG), sd, coder


def cpu_sample(frame):
    """Bounded sample of the workload that keeps its neighbourhood statistics: one quadrant of the scan around the
    sensor (points with x and y at or above the per-axis median), i.e. a spatial crop, not a subsampling -- the
    occupancy of every 3x3x3 neighbourhood inside the crop is the full frame's."""
    c = np.median(frame[:, 1:3], axis=0)
    return np.ascontiguousarray(frame[(frame[:, 1] >= c[0]) & (frame[:, 2] >= c[1])])


def run_reference(args, rank, world):
    """--impl reference: the reference path on the host cores (see cpu_arm_model), all threads, one bounded sample per
    step; under torchrun rank 0 alone runs it."""
    if rank != 0:
        return
    cores = os.cpu_count()
    model, _, coder = cpu_arm_model(cores)
    sample = cpu_sample(make_frames(1, 0)[0])
    times = []
    for i in range(args.warmup + args.steps):
        t = time.perf_counter()
        data = model.compress(sample)
        rec = model.decompress(data)
        dt = time.perf_counter() - t
        assert rec.shape[0] == sample.shape[0]
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [data], [np.ascontiguousarray(rec)])
    ms = 1e3 * sum(times) / len(times)
    v = sample.shape[0] / (ms * 1e-3) / 1e6
    desc = (f'per step: one quadrant of frame 0 of the workload ({sample.shape[0]} pts, spatial crop: same point density), '
            f'compress+decompress; network on torch-CPU SGEMM + OpenMP C element-wise kernels over {cores} threads; {coder}')
    print(json.dumps({
        'impl': 'reference', 'metric': 'encode+decode Mpts/s', 'value': v, 'unit': 'Mpts/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'int8', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'frames_per_step': 0.25, 'sample': desc},
        'cpu_baseline': {'value': v, 'unit': 'Mpts/s', 'cores': cores, 'kind': 'port', 'sample': desc},
        'e2e': {'value': v, 'unit': 'Mpts/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--frames', type=int, default=96, help='frames per step per GPU (coded together, one stream each)')
    ap.add_argument('--groups', type=int, default=3, help='slices of the batch coded concurrently (CUDA streams)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()

    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        if rank == 0:
            os.environ['OMP_NUM_THREADS'] = str(os.cpu_count())  # before torch / libgomp load (torchrun sets it to 1)
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from fastpcc_b200 import _lib, ops, synth
    from fastpcc_b200.lossl_coord_int import Config, Model
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback exists)'
    # Waiting host threads spin by default (lowest latency: 426 ms per step at N = 1) and then hold 2.6 cores per rank (three
    # launching threads); sleeping instead costs 3 % of the step (440 ms) and 0.5 core.  Sleep when the ranks of this job
    # would otherwise claim most of the box's cores (FPCC_SPIN_SYNC=1 / 0 forces either).
    spin = os.environ.get('FPCC_SPIN_SYNC')
    blocking = (spin == '0') if spin in ('0', '1') else (3 * world >= 0.6 * (os.cpu_count() or 1))
    if blocking:
        _lib.load(build_if_missing=False).fpcc_set_blocking_sync(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    _lib.load(build_if_missing=False)

    sd = synth.make_lossl_int_state_dict(seed=7, **CFG)
    model = Model(Config(**CFG), device=dev).load_numpy_state_dict(sd).to(dev)
    frames_host = make_frames(args.frames, rank, world)
    pinned = [torch.from_numpy(f).pin_memory() for f in frames_host]
    frames_dev = [p.to(dev) for p in pinned]
    n_pts = sum(f.shape[0] for f in frames_host)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    G = args.groups

    pipe = os.environ.get('FPCC_BENCH_PIPE', '1') != '0'  # per-group encode -> decode pipelines (Model.roundtrip_batch)

    def step_device():
        """-> (bitstreams, decoded frames)"""
        if pipe:
            return model.roundtrip_batch(frames_dev, n_groups=G)
        data = model.compress_batch(frames_dev, n_groups=G)  # one rANS stream per frame; G slices coded concurrently
        return data, model.decompress_batch(data, n_groups=G)

    h2d = d2h = 0
    host_out = [None]

    def step_e2e():
        nonlocal h2d, d2h
        h2d = d2h = 0
        xs = [p.to(dev, non_blocking=True) for p in pinned]
        if pipe:
            data, rec = model.roundtrip_batch(xs, n_groups=G)  # bytes on the host inside: D2H + H2D of every bitstream
        else:
            data = model.compress_batch(xs, n_groups=G)     # bytes on the host: D2H of the bitstreams inside
            rec = model.decompress_batch(data, n_groups=G)  # H2D of the bitstreams inside
        # D2H of the decoded coordinates: one copy of the concatenated frames into a reused pinned buffer
        cat = torch.cat(rec)
        if host_out[0] is None or host_out[0].shape[0] < cat.shape[0]:
            host_out[0] = torch.empty((cat.shape[0] + (cat.shape[0] >> 3), cat.shape[1]), dtype=cat.dtype, pin_memory=True)
        dst = host_out[0][: cat.shape[0]]
        dst.copy_(cat, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        rec_h = list(dst.split([r.shape[0] for r in rec]))
        nbytes = sum(len(d) for d in data)
        h2d += sum(p.numel() * 4 for p in pinned) + nbytes
        d2h += nbytes + sum(r.numel() * 4 for r in rec_h)
        return rec_h

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_cpu_ms = {}

    def timed(fn, steps, warmup, sample_clocks=False, keep_last=False):
        """-> (ms per step, clocks, what the last step returned if keep_last else None)"""
        for _ in range(warmup):
            fn()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        barrier()
        total_ms = 0.0
        out = None
        cpu0 = time.process_time()  # CPU seconds of ALL threads of this rank: how busy the launching side is
        for i in range(steps):
            flush.fill_(1)  # evict L2 between timed iterations
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if keep_last and i == steps - 1:
                out = fn()
            else:
                fn()
            e1.record()
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
        host_cpu_ms[fn.__name__] = 1e3 * (time.process_time() - cpu0) / steps
        barrier()
        clocks = sampler.summary() if sampler else None
        sys.stderr.write(f'[bench] {fn.__name__}: {steps} steps, {total_ms / steps:.1f} ms/step, host CPU {host_cpu_ms[fn.__name__]:.0f} ms/step, peak mem '
                         f'{torch.cuda.max_memory_allocated() / 2**30:.1f} GiB reserved {torch.cuda.memory_reserved() / 2**30:.1f} GiB\n')
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, clocks, out

    # size-independent property at the full workload: the codec is lossless -- every decoded frame is the input's voxel
    # set (checked once, outside the timed region, on the concurrent-group path that is timed)
    _, rec = step_device()
    lossless = all(torch.equal(torch.unique(r, dim=0), torch.unique(x[:, 1:], dim=0)) for r, x in zip(rec, frames_dev))
    assert lossless, 'decoded frames differ from the input: the measured path is not a valid codec run'
    del rec
    dump = bool(args.dump_outputs) and rank == 0
    ms_dev, clocks, last = timed(step_device, args.steps, args.warmup, sample_clocks=True, keep_last=dump)
    if dump:
        dump_outputs(args.dump_outputs, *last)
    del last
    ms_e2e, _, _ = timed(step_e2e, args.steps, max(1, args.warmup - 1))
    pts_all = torch.tensor([n_pts], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(pts_all)
    pts_all = float(pts_all.item())

    # ---- instrumented pass: CUDA-event time and algorithmic work of every GEMM-class launch -------------
    prof = ops.enable_profile(True)
    model.decompress_batch(model.compress_batch(frames_dev))  # single group: per-launch events on one stream
    torch.cuda.synchronize()
    ops.enable_profile(False)
    stats = ops.profile_summary(prof)
    peaks, peak_kind = load_peaks()
    int8_probe = ops.mma_i8_peak(20000, 256)  # back-to-back tcgen05.mma.kind::i8 on resident tiles, this GPU, now
    # MEASURED_PEAKS.json holds dense bf16 only; kind::i8 issues twice the MACs per instruction.  The conv is timed inside
    # a long step -> the sustained figure.
    peak = 2.0 * float(peaks.get('bf16_tflops_sustained', peaks['bf16_tflops']))
    conv = stats.get('spconv_tc', {'ms': 0.0, 'ops': 0.0, 'launches': 0, 'mma_ops': 0.0})
    traffic = None
    tpath = osp.join(ROOT, 'profiles', 'r02_conv_traffic.json')
    if osp.exists(tpath):  # average DRAM bytes per conv launch of one bench step (ncu, see the file), committed
        with open(tpath) as f:
            traffic = json.load(f)
    roof = {'bound': 'tensor', 'kernel': 'igemm_tc_persistent<CONV> (tcgen05.mma.kind::i8)',
            'achieved': (conv['ops'] / (conv['ms'] * 1e-3) / 1e12) if conv['ms'] else 0.0,
            'peak': peak, 'unit': 'TOP/s', 'traffic': traffic['dram_bytes_per_launch'] if traffic else None,
            'traffic_note': traffic.get('note') if traffic else None,
            'algorithmic_bytes_per_launch': (conv.get('bytes', 0.0) / conv['launches']) if conv['launches'] else None,
            'peak_source': f'2 x bf16_tflops_sustained of MEASURED_PEAKS.json ({peak_kind}): no int8 figure in the file, int8 tcgen05 = 2 x bf16; '
                           f'burst 2 x bf16_tflops = {2.0 * peaks["bf16_tflops"]:.1f}',
            'peak_own_int8_probe': int8_probe,
            'peak_own_note': 'fpcc_mma_i8_peak in this run: tcgen05.mma.kind::i8 M128 N256 K32 back to back on all SMs',
            'launches': conv['launches'], 'ms_per_step': conv['ms'],
            'executed_mma_tops': (conv.get('exec_ops', 0.0) / (conv['ms'] * 1e-3) / 1e12) if conv['ms'] else 0.0,
            'share_of_step': conv['ms'] / ms_dev if ms_dev else 0.0}
    if traffic and roof['algorithmic_bytes_per_launch']:
        # the ncu capture ran the bench's own schedule (launches of frames / groups scans), the instrumented pass one group
        per = traffic.get('frames_per_launch', args.frames) / float(args.frames)
        roof['traffic_over_algorithmic'] = round(traffic['dram_bytes_per_launch'] / (roof['algorithmic_bytes_per_launch'] * per), 2)
    roof['frac_vs_own_probe'] = roof['achieved'] / int8_probe if int8_probe else 0.0
    roof['frac'] = roof['achieved'] / roof['peak'] if roof['peak'] else 0.0
    launches = sum(v['launches'] for v in stats.values())
    # HBM-class kernels (kernel map, coordinate generation, requant, CDF head): algorithmic bytes (SURVEY 8d, stated per
    # wrapper in fastpcc_b200/ops.py) / CUDA-event time of the same instrumented pass, against the measured copy bandwidth
    hbm_peak = float(peaks['hbm_gbs'])
    hbm = {}
    for k, v in stats.items():
        if v.get('bytes') and v['ms'] > 0 and k not in ('spconv_tc', 'linear_tc', 'linear_sel_tc'):
            gbs = v['bytes'] / (v['ms'] * 1e-3) / 1e9
            hbm[k] = {'gb_per_step': round(v['bytes'] / 1e9, 3), 'achieved_gbs': round(gbs, 1), 'frac': round(gbs / hbm_peak, 3)}

    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count()
        om, _, coder = cpu_arm_model(cores)
        sample = cpu_sample(frames_host[0])
        om.compress(sample[: 4096])  # warm-up: thread pools, weight images
        t = time.perf_counter()
        want = om.compress(sample)
        rec = om.decompress(want)
        dt = time.perf_counter() - t
        assert rec.shape[0] == sample.shape[0]
        # parity on the benchmarked configuration (C=256 default topology): the bytes of the CUDA codec against the
        # oracle's on the same sample, alone and inside a batch coded by concurrent groups
        x = torch.from_numpy(sample).to(dev)
        got = model.compress(x)
        batch = model.compress_batch([frames_dev[1], x, frames_dev[2]], n_groups=3)
        dec = model.decompress(got)
        parity = bool(got == want and batch[1] == want and np.array_equal(dec.cpu().numpy(), rec))
        cpu = {'value': sample.shape[0] / dt / 1e6, 'unit': 'Mpts/s', 'cores': cores, 'kind': 'port',
               'sample': f'one quadrant of frame 0 ({sample.shape[0]} pts, spatial crop: same point density), compress+decompress '
                         f'once ({dt:.1f} s); network on torch-CPU SGEMM + OpenMP C element-wise kernels; {coder}'}

    if rank == 0:
        print(json.dumps({
            'metric': 'encode+decode Mpts/s', 'value': pts_all / (ms_dev * 1e-3) / 1e6, 'unit': 'Mpts/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_dev,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int8', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'frames_per_step_per_gpu': args.frames, 'concurrent_groups': G, 'schedule': 'per-group encode->decode pipelines on prioritised streams' if pipe else 'all groups encode, then all groups decode', 'host_sync': 'blocking' if blocking else 'spin', 'points_per_step': pts_all,
                       'l2': 'flushed between timed iterations (256 MB write)', 'weights': 'seeded random int8 (seed 7)',
                       'roundtrip_lossless': bool(lossless), 'parity_sample': parity,
                       'parity_note': 'bitstream of the CUDA codec == bitstream of the CPU oracle (pinned to the reference Python, '
                                      'tests/golden) on the cpu_baseline sample, single and inside a 3-group batch; decoded points equal'},
            'clocks': clocks,
            'e2e': {'value': pts_all / (ms_e2e * 1e-3) / 1e6, 'unit': 'Mpts/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': ms_e2e},
            'gpu_launches': launches * args.steps, 'host_cpu_ms_per_step': round(host_cpu_ms.get('step_device', 0.0), 1),
            'roofline': roof, 'cpu_baseline': cpu,
            'hbm_kernels': {'peak_gbs': hbm_peak, 'peak_source': f'MEASURED_PEAKS.json hbm_gbs ({peak_kind})', 'kernels': hbm},
            'kernels': {k: {'ms': round(v['ms'], 3), 'launches': v['launches']} for k, v in stats.items()},
        }))
    if world > 1:
        dist.destroy_process_group()


def _guarded_main():
    """A failing rank prints its own traceback as its last stderr lines, a one-line JSON {"error": ...} on stdout and a
    copy in a file of its own in the temporary directory, named on stderr (torchrun's failure summary otherwise hides it;
    the tree itself may be read-only); `record` also puts it into that summary."""
    import tempfile
    import traceback
    try:
        from torch.distributed.elastic.multiprocessing.errors import record
        fn = record(main)
    except Exception:
        fn = main
    try:
        fn()
    except SystemExit:
        raise
    except BaseException as e:
        rank = os.environ.get('RANK', '0')
        tb = traceback.format_exc()
        copy = ''
        try:
            fd, path = tempfile.mkstemp(prefix=f'fastpcc_bench_rank{rank}_', suffix='.err')
            with os.fdopen(fd, 'w') as f:
                f.write(tb)
            copy = f' (copy: {path})'
        except OSError:
            pass
        sys.stdout.flush()
        sys.stderr.write(f'\n[bench] rank {rank} FAILED{copy}:\n{tb}\n')
        sys.stderr.flush()
        print(json.dumps({'error': f'rank {rank}: {type(e).__name__}: {e}'[:2000]}), flush=True)
        os._exit(1)


if __name__ == '__main__':
    _guarded_main()
