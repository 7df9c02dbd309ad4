"""The deep-factorized entropy model on the GPU: bits, dy and dparams of the fused kernels against the float64 oracle
(tests/entropy_model_oracle.py), dparams reproducible bit for bit, eval-mode bits at round(y), the coding round trip
through the device tables (escape path included), the stream size against the tables' own code lengths, tables
travelling in the state dict, and LossyColorNet training rate-distortion (bf16, fp16 + GradScaler, both wgrad paths,
DDP replicas)."""
import math
import os

import numpy as np
import pytest
import torch

from tests import entropy_model_oracle as EO

pytestmark = pytest.mark.gpu

# fp32 kernels against fp64 (DESIGN 3.10): bits where L > 1e-6 and their sum to 1e-4 relative; gradients to 1e-3 of
# the largest magnitude (fp32 sigmoid differences and the fp32 sum of the parameter gradient over each thread's rows)
BITS_RTOL, GRAD_RTOL = 1e-4, 1e-3


def _inputs(n, C, seed):
    g = torch.Generator().manual_seed(seed)
    params = EO.random_params(C, g, spread=0.7)
    y = 4.0 * torch.randn((n, C), dtype=torch.float64, generator=g)
    y[: n // 10] *= 250.0                                              # |y| up to ~10^3: the bounded tail
    y[n // 10: n // 5] = torch.randint(-40, 40, (n // 5 - n // 10, C), generator=g).double() + 0.5  # tail and half-integers
    return params, y.float().double()                                  # y exactly representable in fp32


@pytest.mark.parametrize('C', [1, 8, 128])
def test_bits_and_dy_match_the_fp64_oracle(C):
    from fastpcc_b200 import ops
    params, y = _inputs(20000 // C + 37, C, C)
    bits = ops.factorized_bits(y.float().cuda(), params.float().cuda()).double().cpu()
    p32 = params.float().double()                                      # the kernel sees fp32 parameters
    yo = y.clone().requires_grad_()
    ref = EO.bits(p32, yo)
    L = EO.likelihood(p32, y)
    m = L > 1e-6
    rel = ((bits - ref.detach()).abs() / ref.detach().abs().clamp(min=1e-3))[m]
    assert float(rel.max()) < BITS_RTOL, float(rel.max())
    assert abs(float(bits.sum() - ref.detach().sum())) < BITS_RTOL * float(ref.detach().sum())
    bounded = L < 0.5e-9
    assert bool(bounded.any()) and torch.allclose(bits[bounded], torch.full_like(bits[bounded], -math.log2(1e-9)), rtol=1e-6, atol=0)
    g = torch.Generator().manual_seed(3)
    dbits = torch.rand((y.shape[0], C), generator=g, dtype=torch.float64) + 0.5
    (ref * dbits).sum().backward()
    dy, _ = ops.factorized_grad(y.float().cuda(), params.float().cuda(), dbits.float().cuda())
    dy = dy.double().cpu()
    err = (dy - yo.grad)[m].abs().max() / yo.grad[m].abs().max()
    assert float(err) < GRAD_RTOL, float(err)


@pytest.mark.parametrize('n,C', [(3000, 8), (900, 128), (200000, 8)])
def test_dparams_match_autograd_and_are_bit_reproducible(n, C):
    from fastpcc_b200 import ops
    params, y = _inputs(n, C, 11)
    p = params.float().double().requires_grad_()
    g = torch.Generator().manual_seed(4)
    dbits = torch.rand((n, C), generator=g, dtype=torch.float64)
    (EO.bits(p, y) * dbits).sum().backward()
    args = (y.float().cuda(), params.float().cuda(), dbits.float().cuda())
    _, dp1 = ops.factorized_grad(*args)
    _, dp2 = ops.factorized_grad(*args)
    assert torch.equal(dp1, dp2)
    err = (dp1.double().cpu() - p.grad).abs().max() / p.grad.abs().max()
    assert float(err) < GRAD_RTOL, float(err)


def test_module_gradient_reaches_every_parameter():
    from fastpcc_b200.entropy_models import NoisyDeepFactorizedEntropyModel
    torch.manual_seed(0)
    em = NoisyDeepFactorizedEntropyModel(8).cuda()
    y = (3 * torch.randn((5000, 8), device='cuda')).to(torch.bfloat16).requires_grad_()
    y_t, bits = em(y)
    assert y_t.dtype == torch.bfloat16 and bits.dtype == torch.float32
    bits.sum().backward()
    assert y.grad is not None and bool(torch.isfinite(y.grad.float()).all())
    names = dict(em.named_parameters())
    assert sorted(names) == sorted([f'matrices.{i}' for i in range(4)] + [f'biases.{i}' for i in range(4)] +
                                   [f'factors.{i}' for i in range(3)])
    for name, prm in names.items():
        assert prm.grad is not None and float(prm.grad.abs().sum()) > 0, name


def test_eval_mode_bits_at_rounded_values():
    from fastpcc_b200.entropy_models import NoisyDeepFactorizedEntropyModel
    torch.manual_seed(1)
    em = NoisyDeepFactorizedEntropyModel(8).cuda().eval()
    y = 5 * torch.randn((4000, 8), device='cuda')
    y[0, 0], y[1, 0] = 2.5, -1.5                                        # half to even
    with torch.no_grad():
        y_hat, bits = em(y)
    assert torch.equal(y_hat, torch.round(y)) and float(y_hat[0, 0]) == 2.0 and float(y_hat[1, 0]) == -2.0
    ref = EO.bits(em.params().detach().double().cpu(), y_hat.double().cpu())
    m = EO.likelihood(em.params().detach().double().cpu(), y_hat.double().cpu()) > 1e-6
    rel = ((bits.double().cpu() - ref).abs() / ref.abs().clamp(min=1e-3))[m]
    assert float(rel.max()) < BITS_RTOL


def _trained_like(C, seed):
    """a module with perturbed parameters (so channels differ), tables built"""
    from fastpcc_b200.entropy_models import NoisyDeepFactorizedEntropyModel
    torch.manual_seed(seed)
    em = NoisyDeepFactorizedEntropyModel(C).cuda()
    with torch.no_grad():
        for prm in em.parameters():
            prm.add_(0.3 * torch.randn_like(prm))
    em.eval()
    em.update()
    return em


def _host_code_length(em, sym):
    """sum of -log2(freq / 65536) under the stored tables plus the escape bits (sign + Elias-gamma), in bits"""
    flat, off, lens, offs = (t.cpu().numpy() for t in em._tables)
    C = lens.shape[0]
    s = sym.cpu().numpy().reshape(-1, C).astype(np.int64)
    total = 0.0
    for c in range(C):
        cdf = flat[off[c]: off[c] + lens[c]].astype(np.int64)
        maxv = lens[c] - 2
        v = s[:, c] - offs[c]
        esc = (v < 0) | (v >= maxv)
        gamma = np.where(v < 0, -v, v - maxv + 1)
        vc = np.where(esc, maxv, v)
        total += float(-np.log2((cdf[vc + 1] - cdf[vc]) / 65536.0).sum())
        nb = np.floor(np.log2(np.maximum(gamma[esc], 1))).astype(np.int64) + 1
        total += float((2 * nb).sum())
    return total


@pytest.mark.parametrize('C,n', [(1, 1), (1, 1000000), (8, 1), (8, 100000), (128, 1), (128, 3000)])
def test_round_trip_and_stream_size(C, n):
    em = _trained_like(C, 7 + C)
    g = torch.Generator(device='cuda').manual_seed(n + C)
    y = 3 * torch.randn((n, C), device='cuda', generator=g)
    if n > 10:
        y[:: max(1, n // 50)] *= 1000.0                                 # escapes far outside -64 .. 64
        y[5, 0] = -3.0e6
    data = em.compress(y)
    y_hat = em.decompress(data, n)
    assert torch.equal(y_hat, torch.round(y))
    ideal = _host_code_length(em, torch.round(y).to(torch.int32)) / 8
    # 8 bytes of state and flushing, plus the finite-state deviation of rANS (16-bit frequencies, state >= 2^23: each
    # symbol within log2(1 + 2^-7) bits of its ideal length, cancelling on average; DESIGN 3.10)
    assert abs(len(data) - ideal) <= 8 + 1e-4 * ideal, (len(data), ideal)
    if n > 10:
        # the model's own float estimate on in-table symbols: quantising the pmf to 16 bits and the overflow symbol
        # cost at most 2 % + 64 bits (DESIGN 3.10)
        yi = torch.round(y.clamp(-20, 20))
        est = float(em(yi)[1].double().sum())
        got = 8 * len(em.compress(yi))
        print(f'C={C} n={n}: stream {got} bits, model estimate {est:.1f} bits, gap {(got - est) / est:+.4%}')
        assert abs(got - est) <= 0.02 * est + 64, (got, est)


def test_tables_travel_in_the_state_dict():
    from fastpcc_b200.entropy_models import NoisyDeepFactorizedEntropyModel
    em = _trained_like(8, 3)
    flat1 = em._tables[0].clone()
    em.update()
    assert all(torch.equal(a, b) for a, b in zip((flat1,), (em._tables[0],)))  # built twice from the same params
    y = 6 * torch.randn((20000, 8), device='cuda')
    y[::97] *= 200
    data = em.compress(y)
    dec = NoisyDeepFactorizedEntropyModel(8).cuda().eval()
    with pytest.raises(RuntimeError, match='no CDF tables'):
        dec.decompress(data, y.shape[0])
    dec.load_state_dict(em.state_dict())
    assert torch.equal(dec.decompress(data, y.shape[0]), torch.round(y))
    train_mode = NoisyDeepFactorizedEntropyModel(8).cuda()
    with pytest.raises(RuntimeError, match='eval mode'):
        train_mode.update()


# ---------------------------------------------------------------------------------------------------------------------
# LossyColorNet
# ---------------------------------------------------------------------------------------------------------------------
def _train_color(steps, dt, wgrad_tc=True, seed=31):
    from fastpcc_b200 import autograd, me as ME, synth, train
    ME.set_compute_dtype(dt)
    autograd.WGRAD_TC = wgrad_tc
    try:
        torch.manual_seed(0)
        model = train.LossyColorNet(32).cuda()
        opt = torch.optim.Adam(model.parameters(), lr=1e-2)
        scaler = torch.amp.GradScaler('cuda') if dt == torch.float16 else None
        xyz, rgb = synth.colored_surface(seed, bits=8, n_target=40000)
        batch = train.make_color_batch([xyz], [rgb], 'cuda')
        hist = []
        for _ in range(steps):
            loss, terms = train.train_step_color(model, opt, batch, scaler)
            hist.append((float(loss), float(terms['bce']), float(terms['mse']), float(terms['bpp'])))
        return hist, [p.detach().float().clone() for p in model.parameters()]
    finally:
        autograd.WGRAD_TC = True
        ME.set_compute_dtype(torch.float16)


@pytest.mark.parametrize('dt', [torch.float16, torch.bfloat16], ids=['fp16_scaler', 'bf16'])
def test_lossy_color_net_trains_and_wgrad_paths_agree(dt):
    h_tc, p_tc = _train_color(12, dt)
    h_lib, p_lib = _train_color(12, dt, wgrad_tc=False)
    assert np.isfinite(np.array(h_tc)).all(), h_tc
    first, last = h_tc[0], h_tc[-1]
    for k, name in enumerate(['loss', 'bce', 'mse', 'bpp']):
        assert last[k] < first[k], (name, [h[k] for h in h_tc])
    assert abs(h_tc[0][0] - h_lib[0][0]) < 1e-3 and abs(h_tc[-1][0] - h_lib[-1][0]) < 5e-2, (h_tc, h_lib)
    for a, b in zip(p_tc, p_lib):
        assert float((a - b).abs().max()) < 5e-2 * max(1.0, float(b.abs().max()))


def _ddp_worker(rank, world, port, out):
    import torch.distributed as dist
    from fastpcc_b200 import me as ME, synth, train
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', device_id=dev)
    ME.set_compute_dtype(torch.bfloat16)
    torch.manual_seed(0)
    model = train.LossyColorNet(32).to(dev)
    ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[rank])
    opt = torch.optim.Adam(ddp.parameters(), lr=1e-2)
    xyz, rgb = synth.colored_surface(7300 + rank, bits=8, n_target=30000)   # every rank its own coloured cloud
    batch = train.make_color_batch([xyz], [rgb], dev)
    losses = [float(train.train_step_color(ddp, opt, batch)[0]) for _ in range(4)]
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    if rank == 0:
        out.put((losses, float(max((g - gathered[0]).abs().max() for g in gathered))))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_lossy_color_net_ddp_replicas_stay_identical():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, 29647, q)) for r in range(2)]
    for p in procs:
        p.start()
    losses, spread = q.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert spread == 0.0 and losses[-1] < losses[0], (losses, spread)
