"""The Gaussian conditional entropy model and the mean-scale hyperprior on the GPU: bits, dy, dmu and dsigma of the
fused kernels against the float64 oracle (tests/gaussian_oracle.py) with both lower-bound rules, outputs reproducible bit
for bit and equal for column slices, the index rule exactly, the device tables, the coding round trip (escape path
included), the stream size against the tables' code lengths and the model's estimate, tables travelling in the state
dict, the hyperprior's gradients and its decoder, and LossyColorNet training on the hyperprior (bf16, fp16 +
GradScaler, both wgrad paths, DDP replicas)."""
import math
import os

import numpy as np
import pytest
import torch

from tests import gaussian_oracle as GO

pytestmark = pytest.mark.gpu

# fp32 kernels against fp64 (DESIGN 3.11): bits where L > 1e-6 to 1e-4 relative (erfcf differences at sigma <= 300);
# gradients to 1e-3 of the largest magnitude
BITS_RTOL, GRAD_RTOL = 1e-4, 1e-3
# the stream against the model's float estimate at the true sigma, bits per element: rounding sigma up to the next table
# (ratio 1.131: log2 r + (1 / r^2 - 1) / (2 ln 2) = 0.020 bits at large sigma) plus the 16-bit quantisation of the tables
# (at most 0.017 bits per element, the widest table)
EST_OVER, EST_UNDER = 0.04, 0.01


def _inputs(n, C, seed):
    """fp32 y, mu, sigma [n, C]: sigma log-uniform in [0.02, 300] (below the scale bound too), |y - mu| up to 10^3,
    half-integer offsets"""
    g = torch.Generator().manual_seed(seed)
    sigma = torch.exp(torch.empty((n, C), dtype=torch.float64).uniform_(math.log(0.02), math.log(300.0), generator=g))
    mu = 20 * torch.randn((n, C), dtype=torch.float64, generator=g)
    y = mu + sigma * torch.randn((n, C), dtype=torch.float64, generator=g)
    y[: n // 10] = mu[: n // 10] + torch.empty((n // 10, C), dtype=torch.float64).uniform_(-1e3, 1e3, generator=g)
    k = slice(n // 10, n // 5)
    y[k] = torch.round(mu[k]) + torch.randint(-40, 40, y[k].shape, generator=g).double() + 0.5
    mu[k] = torch.round(mu[k])                                         # y - mu a half-integer
    return y.float(), mu.float(), sigma.float()


def _oracle(y, mu, sigma, dbits):
    yo, mo, so = (t.double().requires_grad_() for t in (y, mu, sigma))
    ref = GO.bits(yo, so, mo)
    (ref * dbits.double()).sum().backward()
    return ref.detach(), yo.grad, mo.grad, so.grad


@pytest.mark.parametrize('C', [1, 8, 128])
def test_bits_and_gradients_match_the_fp64_oracle(C):
    from fastpcc_b200 import ops
    y, mu, sigma = _inputs(40000 // C + 37, C, C)
    dbits = torch.rand(y.shape, generator=torch.Generator().manual_seed(3)) + 0.5
    bits = ops.gaussian_bits(y.cuda(), sigma.cuda(), mu.cuda()).double().cpu()
    ref, gy, gm, gs = _oracle(y, mu, sigma, dbits)
    L = GO.likelihood(y.double(), sigma.double(), mu.double())
    m = L > 1e-6
    rel = ((bits - ref).abs() / ref.abs().clamp(min=1e-3))[m]
    assert float(rel.max()) < BITS_RTOL, float(rel.max())
    bounded = L < 0.5e-9
    assert bool(bounded.any()) and torch.allclose(bits[bounded], torch.full_like(bits[bounded], -math.log2(1e-9)), rtol=1e-6, atol=0)
    assert bool((sigma < 0.11).any()) and bool((sigma > 250).any())
    dy, dm, ds = (t.double().cpu() for t in ops.gaussian_grad(y.cuda(), sigma.cuda(), dbits.cuda(), mu.cuda()))
    assert torch.equal(dm, -dy)
    for name, got, want in (('dy', dy, gy), ('dmu', dm, gm), ('dsigma', ds, gs)):
        err = (got - want)[m].abs().max() / want[m].abs().max()
        assert float(err) < GRAD_RTOL, (name, float(err))
    # without means: the mean is 0
    b0 = ops.gaussian_bits((y - mu).cuda(), sigma.cuda()).double().cpu()
    ref0 = GO.bits((y - mu).double(), sigma.double())
    assert float(((b0 - ref0).abs() / ref0.abs().clamp(min=1e-3))[m].max()) < BITS_RTOL


def test_lower_bound_gradient_rules_on_both_sides():
    from fastpcc_b200 import ops
    # likelihood bound: v = 3.75 at sigma = 0.5 (u = -6.5, L ~ 4e-11) is below it while phi(u) is still an fp32 normal,
    # v = 0.3 above; dbits of both signs
    y = torch.tensor([[3.75, 3.75, 0.3, 0.3]], device='cuda')
    s = torch.full_like(y, 0.5)
    db = torch.tensor([[1.0, -1.0, 1.0, -1.0]], device='cuda')
    dy, _, _ = ops.gaussian_grad(y, s, db)
    dy = dy.cpu()[0]
    assert float(dy[0]) > 0 and float(dy[1]) == 0.0      # below the bound: only the step that raises L passes
    assert float(dy[2]) > 0 and float(dy[3]) < 0         # above: both pass
    # scale bound: sigma = 0.02 < 0.11 at v = 1 (a wider scale raises L: passes) and at v = 0 (a narrower one would: stopped)
    y2 = torch.tensor([[1.0, 0.0, 1.0, 0.0]], device='cuda')
    s2 = torch.tensor([[0.02, 0.02, 0.5, 0.5]], device='cuda')
    _, _, ds = ops.gaussian_grad(y2, s2, torch.ones_like(y2))
    ds = ds.cpu()[0]
    assert float(ds[0]) < 0 and float(ds[1]) == 0.0 and float(ds[2]) < 0 and float(ds[3]) > 0
    ref = _oracle(y2.cpu(), torch.zeros_like(y2.cpu()), s2.cpu(), torch.ones_like(y2.cpu()))[3][0]
    assert torch.allclose(ds.double(), ref, rtol=1e-4, atol=1e-7)


def test_outputs_are_reproducible_and_column_slices_equal_copies():
    from fastpcc_b200 import ops
    n, C = 100000, 8
    y, mu, sigma = (t.cuda() for t in _inputs(n, C, 5))
    ms = torch.cat([mu, sigma], 1)                                     # one [n, 2C] tensor, as h_s writes it
    m_sl, s_sl = ms[:, :C], ms[:, C:]
    assert m_sl.stride(0) == 2 * C and not m_sl.is_contiguous()
    db = torch.rand((n, C), device='cuda')
    b1, b2 = ops.gaussian_bits(y, s_sl, m_sl), ops.gaussian_bits(y, s_sl, m_sl)
    assert torch.equal(b1, b2) and torch.equal(b1, ops.gaussian_bits(y, sigma.contiguous(), mu.contiguous()))
    g1, g2 = ops.gaussian_grad(y, s_sl, db, m_sl), ops.gaussian_grad(y, s_sl, db, m_sl)
    g3 = ops.gaussian_grad(y, sigma.contiguous(), db, mu.contiguous())
    for a, b, c in zip(g1, g2, g3):
        assert torch.equal(a, b) and torch.equal(a, c)
    i1 = ops.gaussian_indexes(torch.tensor([0.11, 1.0, 10.0], device='cuda'), s_sl, m_sl, y)
    i2 = ops.gaussian_indexes(torch.tensor([0.11, 1.0, 10.0], device='cuda'), sigma.contiguous(), mu.contiguous(), y)
    assert torch.equal(i1[0], i2[0]) and torch.equal(i1[1], i2[1])


def test_autograd_reaches_y_scales_and_means_in_the_compute_dtype():
    from fastpcc_b200 import autograd
    y, mu, sigma = (t.cuda().to(torch.bfloat16).requires_grad_() for t in _inputs(3000, 8, 9))
    bits = autograd.gaussian_bits(y, sigma, mu)
    assert bits.dtype == torch.float32
    bits.sum().backward()
    for t in (y, mu, sigma):
        assert t.grad is not None and t.grad.dtype == torch.bfloat16 and bool(torch.isfinite(t.grad.float()).all())
        assert float(t.grad.float().abs().sum()) > 0


def test_indexes_and_symbols_follow_the_rule_exactly():
    from fastpcc_b200 import ops
    from fastpcc_b200.entropy_models import default_scale_table
    table = default_scale_table()
    t_up = torch.nextafter(table, torch.full_like(table, 1e9))
    t_dn = torch.nextafter(table, torch.zeros_like(table))
    g = torch.Generator().manual_seed(2)
    rnd = torch.exp(torch.empty(20000, dtype=torch.float64).uniform_(math.log(0.01), math.log(400.0), generator=g)).float()
    sigma = torch.cat([table, t_up, t_dn, rnd, torch.tensor([0.0, -3.0, 1e30])]).reshape(-1, 1).repeat(1, 3).contiguous()
    n = sigma.shape[0]
    mu = torch.randn((n, 3), generator=g) * 50
    y = mu + torch.randn((n, 3), generator=g) * 20
    y[:64, 0] = mu[:64, 0] + torch.arange(-32, 32).float() + 0.5     # half to even
    sym, idx = ops.gaussian_indexes(table.cuda(), sigma.cuda(), mu.cuda(), y.cuda())
    assert torch.equal(idx.cpu().long(), GO.indexes(sigma, table))
    assert torch.equal(sym.cpu(), torch.round(y - mu).to(torch.int32))
    idx2 = ops.gaussian_indexes(table.cuda(), sigma.cuda())             # the decoder's call: same indexes
    assert torch.equal(idx, idx2)


def _built(seed=0, **kw):
    from fastpcc_b200.entropy_models import GaussianConditionalEntropyModel
    em = GaussianConditionalEntropyModel(**kw).cuda().eval()
    em.update()
    return em


def test_tables_match_their_centers_and_the_float_pmf():
    from fastpcc_b200 import ops
    em = _built()
    flat1 = em._tables[0].clone()
    em.update()
    assert all(torch.equal(a, b) for a, b in zip((flat1,), (em._tables[0],)))      # built twice: the same tables
    table = em.scale_table.cpu()
    centers = ops.gaussian_centers(em.scale_table).tolist()
    assert centers[-1] == 1565
    pmf, offs = ops.gaussian_pmf(em.scale_table)
    assert pmf.shape == (64, 3131) and offs.cpu().tolist() == [-c for c in centers]
    want = GO.pmf_rows(table.double(), centers)
    assert float((pmf.cpu() - want).abs().max()) < 2e-6
    flat, off, lens, offsets = (t.cpu().numpy().astype(np.int64) for t in em._tables)
    for t, c in enumerate(centers):
        cdf = flat[off[t]: off[t] + lens[t]]
        nin = lens[t] - 2                                              # in-table symbols; the last entry is the escape
        assert -c <= offsets[t] and offsets[t] + nin - 1 <= c, (t, c, offsets[t], nin)
        p = want[t, :2 * c + 1].numpy()
        k = np.arange(-c, c + 1)
        assert (p[(k < offsets[t]) | (k >= offsets[t] + nin)] < 2.0 / 65536).all()   # only negligible symbols escape
        freq = np.diff(cdf)
        assert cdf[0] == 0 and cdf[-1] == 65536 and (freq >= 1).all()
        inside = (k >= offsets[t]) & (k < offsets[t] + nin)
        cost = np.empty_like(p)
        cost[inside] = -np.log2(freq[k[inside] - offsets[t]] / 65536.0)
        v = k[~inside] - offsets[t]
        gamma = np.where(v < 0, -v, v - nin + 1)
        cost[~inside] = -np.log2(freq[nin] / 65536.0) + 2 * (np.floor(np.log2(np.maximum(gamma, 1))) + 1)
        H = -(p * np.log2(np.where(p > 0, p, 1))).sum()
        X = (p * cost).sum()
        # ideal code length under the quantised table within 0.02 bits per element of the float pmf's entropy
        assert -1e-9 <= X - H < 0.02, (t, float(table[t]), H, X)


def _host_code_length(em, sym, idx):
    """sum of -log2(freq / 65536) under the stored tables plus the escape bits (sign + Elias-gamma), in bits"""
    flat, off, lens, offs = (t.cpu().numpy().astype(np.int64) for t in em._tables)
    s, i = sym.cpu().numpy().reshape(-1).astype(np.int64), idx.cpu().numpy().reshape(-1).astype(np.int64)
    maxv = lens[i] - 2
    v = s - offs[i]
    esc = (v < 0) | (v >= maxv)
    gamma = np.where(v < 0, -v, v - maxv + 1)
    vc = np.where(esc, maxv, v)
    base = off[i]
    freq = flat[base + vc + 1] - flat[base + vc]
    nb = np.floor(np.log2(np.maximum(gamma[esc], 1))).astype(np.int64) + 1
    return float(-np.log2(freq / 65536.0).sum()) + float((2 * nb).sum())


@pytest.mark.parametrize('C,n', [(1, 1), (1, 1000000), (8, 1), (8, 125000), (128, 1), (128, 7813)])
def test_round_trip_and_stream_size(C, n):
    from fastpcc_b200 import ops
    em = _built()
    g = torch.Generator(device='cuda').manual_seed(n + C)
    sigma = torch.exp(torch.empty((n, C), device='cuda').uniform_(math.log(0.05), math.log(300.0), generator=g))
    mu = 30 * torch.randn((n, C), device='cuda', generator=g)
    y = mu + sigma * torch.randn((n, C), device='cuda', generator=g)
    if n > 10:
        y[:: max(1, n // 50)] += 1.0e5                                 # escapes far outside the widest table (+-1565)
        y[5, 0] = -3.0e6
    data = em.compress(y, sigma, mu)
    y_hat = em.decompress(data, sigma, mu)
    assert torch.equal(y_hat, torch.round(y - mu) + mu)
    sym, idx = ops.gaussian_indexes(em.scale_table, sigma, mu, y)
    ideal = _host_code_length(em, sym, idx) / 8
    # 8 bytes of state and flushing, plus the finite-state deviation of rANS (DESIGN 3.10)
    assert abs(len(data) - ideal) <= 8 + 1e-4 * ideal, (len(data), ideal)
    if n > 10:
        # in-table symbols against the model's own float estimate at the true sigma
        yi = mu + torch.maximum(torch.minimum(y - mu, 3 * sigma), -3 * sigma)
        est = float(em(yi, sigma, mu)[1].double().sum())
        got = 8 * len(em.compress(yi, sigma, mu))
        print(f'C={C} n={n}: stream {got} bits, model estimate {est:.1f} bits, {(got - est) / (n * C):+.4f} bits per element')
        assert -EST_UNDER * n * C - 64 <= got - est <= EST_OVER * n * C + 64, (got, est)


def test_tables_travel_in_the_state_dict():
    from fastpcc_b200.entropy_models import GaussianConditionalEntropyModel
    em = _built()
    n, C = 20000, 8
    sigma = torch.rand((n, C), device='cuda') * 20
    mu = torch.randn((n, C), device='cuda')
    y = mu + 3 * sigma * torch.randn((n, C), device='cuda')
    y[::97] *= 300
    data = em.compress(y, sigma, mu)
    dec = GaussianConditionalEntropyModel().cuda().eval()
    with pytest.raises(RuntimeError, match='no CDF tables'):
        dec.decompress(data, sigma, mu)
    dec.load_state_dict(em.state_dict())
    assert torch.equal(dec.decompress(data, sigma, mu), torch.round(y - mu) + mu)
    with pytest.raises(RuntimeError, match='eval mode'):
        GaussianConditionalEntropyModel().cuda().update()


def test_eval_forward_dequantises_around_the_mean():
    em = _built()
    y, mu, sigma = (t.cuda() for t in _inputs(4000, 8, 12))
    with torch.no_grad():
        y_hat, bits = em(y, sigma, mu)
    assert torch.equal(y_hat, torch.round(y - mu) + mu)
    ref = GO.bits(y_hat.double().cpu(), sigma.double().cpu(), mu.double().cpu())
    m = GO.likelihood(y_hat.double().cpu(), sigma.double().cpu(), mu.double().cpu()) > 1e-6
    assert float(((bits.double().cpu() - ref).abs() / ref.abs().clamp(min=1e-3))[m].max()) < BITS_RTOL


# ---------------------------------------------------------------------------------------------------------------------
# HyperpriorEntropyModel
# ---------------------------------------------------------------------------------------------------------------------
def _latent(seed, latent, device='cuda', n_target=30000):
    """a stride-2 latent on a synthetic surface: (coords int32 [n, 4] Morton ordered, features [n, latent])"""
    from fastpcc_b200 import me as ME, synth
    xyz = synth.surface_cloud(seed, bits=9, n_target=n_target)
    c = torch.from_numpy(synth.with_batch(xyz)).to(device).to(torch.int32)
    c[:, 1:] = torch.div(c[:, 1:], 2, rounding_mode='floor') * 2
    c = torch.unique(c, dim=0)
    c = c[ME.morton_order(c, 2)].contiguous()
    g = torch.Generator(device=device).manual_seed(seed)
    return c, 4 * torch.randn((c.shape[0], latent), device=device, generator=g)


def test_hyperprior_gradient_reaches_every_parameter():
    from fastpcc_b200 import me as ME
    from fastpcc_b200.entropy_models import HyperpriorEntropyModel
    ME.set_compute_dtype(torch.bfloat16)
    try:
        torch.manual_seed(0)
        hp = HyperpriorEntropyModel(8, 8, 32).cuda()
        c, f = _latent(3, 8)
        f = f.to(torch.bfloat16).requires_grad_()
        y = ME.SparseTensor(f, coordinates=c, tensor_stride=2)
        y_t, bits_y, bits_z = hp(y)
        assert y_t.coordinate_map_key == y.coordinate_map_key and y_t.F.dtype == torch.bfloat16
        assert bits_y.shape == (c.shape[0], 8) and bits_z.shape[1] == 8 and bits_z.shape[0] < c.shape[0]
        (bits_y.sum() + bits_z.sum() + y_t.F.float().square().sum()).backward()
        assert f.grad is not None and bool(torch.isfinite(f.grad.float()).all())
        for name, prm in hp.named_parameters():
            assert prm.grad is not None and bool(torch.isfinite(prm.grad).all()) and float(prm.grad.abs().sum()) > 0, name
    finally:
        ME.set_compute_dtype(torch.float16)


@pytest.mark.parametrize('dt', [torch.float16, torch.bfloat16], ids=['fp16', 'bf16'])
def test_hyperprior_decodes_from_coordinates_only(dt):
    from fastpcc_b200 import me as ME
    from fastpcc_b200.entropy_models import HyperpriorEntropyModel
    ME.set_compute_dtype(dt)
    try:
        torch.manual_seed(1)
        enc = HyperpriorEntropyModel(8, 8, 32).cuda()
        c, f = _latent(4, 8)
        y = ME.SparseTensor(f.to(dt), coordinates=c, tensor_stride=2)
        enc(y)[1].sum().backward()                                     # a training step's worth of state, then eval
        enc.eval()
        enc.update()
        data = enc.compress(y)
        with torch.no_grad():
            z = enc.h_a_mlp(enc.h_a_conv(y))
            mu, sigma = enc.means_scales(z._like(torch.round(z.F.float()).to(dt)), y.coordinate_map_key)
            want = torch.round(y.F.float() - mu) + mu
            y_eval, _, _ = enc(y)
        assert torch.equal(y_eval.F, want.to(dt))
        dec = HyperpriorEntropyModel(8, 8, 32).cuda().eval()
        dec.load_state_dict(enc.state_dict())
        skeleton = ME.SparseTensor(torch.zeros((c.shape[0], 1), device='cuda'), coordinates=c.clone(), tensor_stride=2)
        y_hat = dec.decompress(data, skeleton)
        assert y_hat.coordinate_map_key == skeleton.coordinate_map_key
        assert y_hat.F.dtype == torch.float32 and torch.equal(y_hat.F, want)
        print(f'{dt}: {c.shape[0]} x 8 latent -> {len(data)} bytes ({8 * len(data) / c.shape[0]:.2f} bits per latent row)')
    finally:
        ME.set_compute_dtype(torch.float16)


# ---------------------------------------------------------------------------------------------------------------------
# LossyColorNet on the hyperprior
# ---------------------------------------------------------------------------------------------------------------------
def _train_color(steps, dt, wgrad_tc=True, seed=31):
    from fastpcc_b200 import autograd, me as ME, synth, train
    ME.set_compute_dtype(dt)
    autograd.WGRAD_TC = wgrad_tc
    try:
        torch.manual_seed(0)
        model = train.LossyColorNet(32, prior='hyperprior').cuda()
        opt = torch.optim.Adam(model.parameters(), lr=1e-2)
        scaler = torch.amp.GradScaler('cuda') if dt == torch.float16 else None
        xyz, rgb = synth.colored_surface(seed, bits=8, n_target=40000)
        batch = train.make_color_batch([xyz], [rgb], 'cuda')
        hist = []
        for _ in range(steps):
            loss, terms = train.train_step_color(model, opt, batch, scaler)
            assert sorted(terms) == ['bce', 'bpp', 'mse']
            hist.append((float(loss), float(terms['bce']), float(terms['mse']), float(terms['bpp'])))
        return hist, [p.detach().float().clone() for p in model.parameters()]
    finally:
        autograd.WGRAD_TC = True
        ME.set_compute_dtype(torch.float16)


@pytest.mark.parametrize('dt', [torch.float16, torch.bfloat16], ids=['fp16_scaler', 'bf16'])
def test_lossy_color_net_hyperprior_trains_and_wgrad_paths_agree(dt):
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
    model = train.LossyColorNet(32, prior='hyperprior').to(dev)
    ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[rank])
    opt = torch.optim.Adam(ddp.parameters(), lr=1e-2)
    xyz, rgb = synth.colored_surface(7400 + rank, bits=8, n_target=30000)   # every rank its own coloured cloud
    batch = train.make_color_batch([xyz], [rgb], dev)
    losses = [float(train.train_step_color(ddp, opt, batch)[0]) for _ in range(4)]
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    if rank == 0:
        out.put((losses, float(max((g - gathered[0]).abs().max() for g in gathered))))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_lossy_color_net_hyperprior_ddp_replicas_stay_identical():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, 29651, q)) for r in range(2)]
    for p in procs:
        p.start()
    losses, spread = q.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert spread == 0.0 and losses[-1] < losses[0], (losses, spread)
