"""Gradients through the MinkowskiEngine shim on the GPU: the transposed neighbour table (fpcc_kmap_transpose) and the
fused-activation backward (fpcc_act_grad_f16) against their torch references; every layer kind's output, d_feats,
d_kernel and d_bias against torch autograd through the dense fp64 restatement of tests/me_grad_oracle.py; the forward
bits do not depend on the grad mode; LossyGeoNet trains in bf16 and in fp16 with a GradScaler, on the tensor-core
wgrad and on the per-offset library GEMMs alike; with two GPUs DistributedDataParallel keeps its replicas identical."""
import os

import numpy as np
import pytest
import torch

from tests import me_grad_oracle as MO

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
TOL = {torch.float16: 1e-2, torch.bfloat16: 4e-2}


@pytest.fixture
def me_dtype():
    from fastpcc_b200 import me as ME
    yield ME
    ME.set_compute_dtype(torch.float16)


def _coords(xyz, device='cuda'):
    from fastpcc_b200 import train
    return train.make_lossy_batch([xyz], device)


def _surface(n=10000, seed=3):
    from fastpcc_b200 import synth
    return synth.surface_cloud(seed, bits=7, n_target=n)


# ---------------------------------------------------------------------------------------------------------------------
# fpcc_kmap_transpose
# ---------------------------------------------------------------------------------------------------------------------
def _maps(xyz):
    """(name, table, n_in): k3 stride 1, k2s2, k3 onto an explicit coarser key, transposed-conv slot table with orphans"""
    from fastpcc_b200 import me as ME, ops
    x = ME.SparseTensor(torch.ones((xyz.shape[0], 1), device='cuda'), coordinates=_coords(xyz))
    cm, k1 = x.coordinate_manager, x.coordinate_map_key
    k2 = cm.stride(k1, 2)
    n1, n2 = cm.get_coordinates(k1).shape[0], cm.get_coordinates(k2).shape[0]
    out = [('k3s1', cm.kernel_table(k1, k1, 3, (1, 1, 1)), n1),
           ('k2s2', cm.kernel_table(k1, k2, 2, (1, 1, 1)), n1),
           ('k3_onto_coarse', cm.kernel_table(k1, k2, 3, (1, 1, 1)), n1)]
    # parents: every other stride-2 voxel, so the children of the dropped ones are orphans (slot 255, no table entry)
    pc = cm.get_coordinates(k2)[::2].contiguous()
    keys, vals = ops.hash_build(pc)
    fine = cm.get_coordinates(k1)
    par_c = fine.clone()
    par_c[:, 1:] = torch.div(fine[:, 1:], 2, rounding_mode='floor') * 2
    par = ops.kmap_lookup(keys, vals, par_c.contiguous(), (1, 1, 1), (1, 1, 1), convention=1)[0] - 1
    d = fine[:, 1:] - par_c[:, 1:]
    slot = (d[:, 0] + 2 * d[:, 1] + 4 * d[:, 2]).to(torch.uint8)
    slot = torch.where(par >= 0, slot, torch.full_like(slot, 255))
    assert bool((par < 0).any()) and bool((par >= 0).any())
    out.append(('slot_table_orphans', ops.slot_table(par.clamp(min=0).contiguous(), slot.contiguous()), pc.shape[0]))
    return out


@pytest.mark.parametrize('cloud', ['surface', 'lidar', 'surface_1M'])
def test_kmap_transpose_equals_the_torch_scatter(cloud):
    from fastpcc_b200 import ops, synth
    if cloud == 'surface':
        xyz = synth.surface_cloud(11, bits=10, n_target=200000)
    elif cloud == 'lidar':
        xyz = synth.lidar_frame(5)
    else:
        xyz = synth.surface_cloud(12, bits=11, n_target=1 << 21)
    assert cloud != 'surface_1M' or xyz.shape[0] >= 1 << 20
    for name, table, n_in in _maps(xyz):
        tt = ops.kmap_transpose(table, n_in)
        assert torch.equal(tt, MO.transpose_table(table, n_in)), name
        assert torch.equal(ops.kmap_transpose(tt, table.shape[1]), table) or name.startswith('slot'), name


# ---------------------------------------------------------------------------------------------------------------------
# fpcc_act_grad_f16
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('act,slope', [(MO.ACT_RELU, 0.0), (MO.ACT_LEAKY, 0.2), (MO.ACT_NONE, 0.0)])
@pytest.mark.parametrize('dy_dt', [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize('y_dt', [torch.float16, torch.bfloat16, torch.float32])
def test_act_grad_is_exact_and_dbias_reproducible(act, slope, dy_dt, y_dt):
    from fastpcc_b200 import ops
    g = torch.Generator(device='cuda').manual_seed(1)
    n, c, c_pad = 100003, 13, 16
    dy = torch.randn((n, c), device='cuda', generator=g).to(dy_dt)
    y = torch.randn((n, c), device='cuda', generator=g).to(y_dt)
    y[::7, 3] = 0  # exact zeros take the slope branch
    for dz_dt in DTYPES:
        dz, db = ops.act_grad_f16(dy, y, act, slope, c_pad, out_dtype=dz_dt)
        ref, ref_db = MO.act_grad(dy, y, act, slope, c_pad, dz_dt)
        assert dz.dtype == dz_dt and torch.equal(dz, ref)
        assert bool((dz[:, c:] == 0).all())
        bound = 1e-6 * ref_db.abs() + 1e-12 * (dy.double().abs().sum(0))
        assert bool(((db.double() - ref_db).abs() <= bound).all()), (db, ref_db)
        dz2, db2 = ops.act_grad_f16(dy, y, act, slope, c_pad, out_dtype=dz_dt)
        assert torch.equal(db2.view(torch.int32), db.view(torch.int32)) and torch.equal(dz2, dz)


def test_act_grad_reads_a_strided_forward_output():
    """the layers keep a column slice of the padded kernel output as Y"""
    from fastpcc_b200 import ops
    g = torch.Generator(device='cuda').manual_seed(2)
    y_full = torch.randn((5000, 16), device='cuda', generator=g).half()
    dy = torch.randn((5000, 10), device='cuda', generator=g).half()
    dz, db = ops.act_grad_f16(dy, y_full[:, :10], MO.ACT_RELU, 0.0, 16)
    ref, ref_db = MO.act_grad(dy, y_full[:, :10].contiguous(), MO.ACT_RELU, 0.0, 16, torch.float16)
    assert torch.equal(dz, ref) and float((db.double() - ref_db).abs().max()) <= 1e-6 * float(ref_db.abs().max())


# ---------------------------------------------------------------------------------------------------------------------
# per layer kind against torch autograd through the fp64 restatement
# ---------------------------------------------------------------------------------------------------------------------
def _rel(a, b):
    return float((a.double().cpu() - b.double().cpu()).abs().max()) / max(float(b.double().abs().max()), 1e-30)


def _case(name, ME, L, dt, seed=0):
    """-> (block, input SparseTensor, extra forward args, reference fn(f64, params64 dict, m) -> out64).  m(module name)
    is the sign mask (Y > 0) of that conv / linear block's forward output under test: the reference takes the
    activation's branch from it, so a pre-activation within rounding of the kink cannot flip a whole dY entry."""
    torch.manual_seed(seed)
    xyz = _surface()
    coords = _coords(xyz)
    g = torch.Generator(device='cuda').manual_seed(seed + 100)

    def inp(c_in, key=None, cm=None):
        if key is None:
            x = ME.SparseTensor(torch.randn((coords.shape[0], c_in), device='cuda', generator=g).to(dt), coordinates=coords)
        else:
            n = cm.get_coordinates(key).shape[0]
            x = ME.SparseTensor(torch.randn((n, c_in), device='cuda', generator=g).to(dt), coordinate_map_key=key, coordinate_manager=cm)
        x.F.requires_grad_()
        return x

    def tab(x, out_key, ks, scale=1):
        cm = x.coordinate_manager
        return MO.table(cm.get_coordinates(x.coordinate_map_key), cm.get_coordinates(out_key), ks, scale)

    R, LK = MO.ACT_RELU, MO.ACT_LEAKY
    if name in ('k3s1', 'k3s1_noact', 'k2s2', 'k3_onto_coarse', 'conv1x1', 'prelu', 'bn_prelu'):
        c_out = 24
        if name == 'k3s1':
            blk = L.ConvBlock(16, c_out, 3, 1, act='relu')
        elif name == 'k3s1_noact':
            blk = L.ConvBlock(16, c_out, 3, 1, act=None)
        elif name == 'k2s2':
            blk = L.ConvBlock(16, c_out, 2, 2, act='leaky_relu(0.2)')
        elif name == 'k3_onto_coarse':
            blk = L.ConvBlock(16, c_out, 3, 2, act='relu')
        elif name == 'conv1x1':
            blk = L.ConvBlock(16, c_out, 1, 1, act='relu')
        elif name == 'prelu':
            blk = L.ConvBlock(16, c_out, 3, 1, act='prelu')
        else:
            blk = L.ConvBlock(16, c_out, 3, 1, bn=True, act='prelu')
        blk = blk.cuda()
        x = inp(16)
        cm = x.coordinate_manager
        args = ()
        if name == 'k3_onto_coarse':
            out_key = cm.stride(x.coordinate_map_key, 2)
            args = (out_key,)
        elif name == 'k2s2':
            out_key = cm.stride(x.coordinate_map_key, 2)
        else:
            out_key = x.coordinate_map_key
        ks = blk.conv.kernel_generator.kernel_size
        t = tab(x, out_key, ks)

        def ref(f, p, m):
            w = p['conv.kernel']
            w = w[None] if w.dim() == 2 else w
            b = p.get('conv.bias')
            code, slope = {'k3s1': (R, 0.0), 'k2s2': (LK, 0.2), 'k3_onto_coarse': (R, 0.0), 'conv1x1': (R, 0.0)}.get(name, (0, 0.0))
            y = MO.conv(f, w, b, t, code, slope, m('') if code else None)
            if name == 'bn_prelu':
                mu, var = y.mean(0, keepdim=True), y.var(0, unbiased=False, keepdim=True)
                y = (y - mu) / torch.sqrt(var + 1e-5) * p['bn.bn.weight'] + p['bn.bn.bias']
            if name in ('prelu', 'bn_prelu'):
                y = torch.where(y > 0, y, y * p['act_module.weight'])
            return y
        return blk, x, args, ref
    if name == 'linear':
        blk = L.MEMLPBlock(16, 8).cuda()
        x = inp(16)
        return blk, x, (), lambda f, p, m: MO.act(f @ p['mlp.linear.weight'].t() + p['mlp.linear.bias'], R, 0.0, m(''))
    if name == 'gen':
        blk = L.GenConvTransBlock(32, 16, 2, 2, act='relu').cuda()
        x0 = inp(1)
        k2 = x0.coordinate_manager.stride(x0.coordinate_map_key, 2)
        x = inp(32, k2, x0.coordinate_manager)
        return blk, x, (), lambda f, p, m: MO.gen(f, p['conv.kernel'], p['conv.bias'], R, mask=m(''))
    if name == 'tconv':
        blk = L.ConvTransBlock(32, 16, 2, 2, act='leaky_relu(0.2)').cuda()
        x0 = inp(1)
        cm = x0.coordinate_manager
        k2 = cm.stride(x0.coordinate_map_key, 2)
        keep = torch.arange(cm.get_coordinates(k2).shape[0], device='cuda') % 3 != 0  # dropped parents leave orphans
        xp = ME.MinkowskiPruning()(ME.SparseTensor(torch.zeros((keep.shape[0], 1), device='cuda'), coordinate_map_key=k2,
                                                   coordinate_manager=cm), keep)
        x = inp(32, xp.coordinate_map_key, cm)
        in_c, out_c = cm.get_coordinates(x.coordinate_map_key), cm.get_coordinates(x0.coordinate_map_key)
        return blk, x, (x0.coordinate_map_key,), lambda f, p, m: MO.tconv(f, p['conv.kernel'], p['conv.bias'], in_c, out_c, 2, LK, 0.2, m(''))
    if name in ('res', 'inception'):
        ch = 32
        blk = (L.ResBlock(ch, 'HYPER_CUBE', False, 'relu') if name == 'res' else L.InceptionResBlock(ch, 'HYPER_CUBE', False, 'relu')).cuda()
        x = inp(ch)
        key = x.coordinate_map_key
        t3, t1 = tab(x, key, (3, 3, 3)), tab(x, key, (1, 1, 1))

        def ref(f, p, m):
            def cb(f, pre, t, code):
                w = p[pre + '.conv.kernel']
                return MO.conv(f, w if w.dim() == 3 else w[None], p[pre + '.conv.bias'], t, code, mask=m(pre) if code else None)

            if name == 'res':
                return cb(cb(f, 'conv0', t3, R), 'conv1', t3, 0) + f
            a = cb(cb(f, 'path_0.0', t3, R), 'path_0.1', t3, 0)
            b = cb(cb(cb(f, 'path_1.0', t1, R), 'path_1.1', t3, R), 'path_1.2', t1, 0)
            return torch.cat([a, b], 1) + f
        return blk, x, (), ref
    raise KeyError(name)


LAYERS = ['k3s1', 'k3s1_noact', 'k2s2', 'k3_onto_coarse', 'conv1x1', 'linear', 'gen', 'tconv', 'res', 'inception',
          'prelu', 'bn_prelu']


@pytest.mark.parametrize('dt', DTYPES, ids=['fp16', 'bf16'])
@pytest.mark.parametrize('name', LAYERS)
def test_layer_gradients_match_fp64_autograd(name, dt, me_dtype):
    from fastpcc_b200 import minkowski_sparse_conv_layers as L
    ME = me_dtype
    ME.set_compute_dtype(dt)
    blk, x, args, ref = _case(name, ME, L, dt)
    assert x.F.shape[0] >= ME.GROUP_ROWS_MIN or name in ('gen', 'tconv')  # grouped forward and dgrad tables
    seen = {}
    hooks = [mod.register_forward_hook(lambda mod, i, o, n=n: seen.__setitem__(n, o.F.detach()))
             for n, mod in blk.named_modules() if isinstance(mod, (L.BaseConvBlock, L.MEMLPBlock))]
    out = blk(x, *args).F
    for h in hooks:
        h.remove()
    r = torch.randn(out.shape, device='cuda', generator=torch.Generator(device='cuda').manual_seed(9))
    (out.float() * r).sum().backward()
    f64 = x.F.detach().double().cpu().requires_grad_()
    # conv / linear weights as the kernels multiply them (rounded to the compute dtype); biases, batch norm and the
    # PReLU slope are used unrounded on the fp32 side
    p64 = {n: (p.detach().to(dt) if n.endswith(('kernel', 'linear.weight')) else p.detach()).double().cpu().requires_grad_()
           for n, p in blk.named_parameters()}
    o64 = ref(f64, p64, lambda n: (seen[n].float() > 0).cpu())
    (o64 * r.double().cpu()).sum().backward()
    tol = TOL[dt]
    assert out.shape == o64.shape
    assert _rel(out.detach(), o64.detach()) < tol, ('out', _rel(out.detach(), o64.detach()))
    assert x.F.grad is not None and _rel(x.F.grad, f64.grad) < tol, ('d_feats', _rel(x.F.grad, f64.grad))
    for n, p in blk.named_parameters():
        assert p.grad is not None and p.grad.dtype == torch.float32, n
        assert _rel(p.grad, p64[n].grad) < tol, (n, _rel(p.grad, p64[n].grad))


@pytest.mark.parametrize('dt', DTYPES, ids=['fp16', 'bf16'])
@pytest.mark.parametrize('name', [n for n in LAYERS if n not in ('prelu', 'bn_prelu')])
def test_grad_mode_does_not_change_the_forward(name, dt, me_dtype):
    """PReLU blocks are left out on purpose: inference fuses the slope into the epilogue, training applies it after"""
    from fastpcc_b200 import minkowski_sparse_conv_layers as L
    ME = me_dtype
    ME.set_compute_dtype(dt)
    blk, x, args, _ = _case(name, ME, L, dt)
    with torch.no_grad():
        a = blk(x, *args).F
    b = blk(x, *args).F
    assert b.requires_grad and torch.equal(a, b.detach())


# ---------------------------------------------------------------------------------------------------------------------
# training
# ---------------------------------------------------------------------------------------------------------------------
def _train(steps, dt, wgrad_tc=True, seed=21):
    from fastpcc_b200 import autograd, me as ME, synth, train
    ME.set_compute_dtype(dt)
    autograd.WGRAD_TC = wgrad_tc
    try:
        torch.manual_seed(0)
        model = train.LossyGeoNet(32).cuda()
        opt = torch.optim.Adam(model.parameters(), lr=1e-2)
        scaler = torch.amp.GradScaler('cuda') if dt == torch.float16 else None
        batch = train.make_lossy_batch([synth.surface_cloud(seed, bits=8, n_target=40000)], 'cuda')
        slope0 = float(model.tconv.act_module.weight.detach().item())
        losses = []
        for i in range(steps):
            losses.append(float(train.train_step_lossy(model, opt, batch, scaler)))
            if i == 0:
                slope1 = float(model.tconv.act_module.weight.detach().item())
        return losses, [p.detach().float().clone() for p in model.parameters()], (slope0, slope1)
    finally:
        autograd.WGRAD_TC = True
        ME.set_compute_dtype(torch.float16)


@pytest.mark.parametrize('dt', DTYPES, ids=['fp16_scaler', 'bf16'])
def test_lossy_geo_net_trains_and_wgrad_paths_agree(dt):
    l_tc, p_tc, (s0, s1) = _train(6, dt)
    l_lib, p_lib, _ = _train(6, dt, wgrad_tc=False)
    assert all(np.isfinite(l_tc)) and l_tc[-1] < l_tc[0] - 0.05, l_tc
    if dt == torch.bfloat16:  # (fp16: the GradScaler may skip the first step while it finds its scale)
        assert s1 != s0, 'the PReLU slope did not train'
    assert abs(l_tc[0] - l_lib[0]) < 1e-3 and abs(l_tc[-1] - l_lib[-1]) < 5e-2, (l_tc, l_lib)
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
    model = train.LossyGeoNet(32).to(dev)
    ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[rank])
    opt = torch.optim.Adam(ddp.parameters(), lr=1e-2)
    batch = train.make_lossy_batch([synth.surface_cloud(7200 + rank, bits=8, n_target=30000)], dev)  # every rank its own cloud
    losses = [float(train.train_step_lossy(ddp, opt, batch)) for _ in range(4)]
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    if rank == 0:
        out.put((losses, float(max((g - gathered[0]).abs().max() for g in gathered))))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_lossy_geo_net_ddp_replicas_stay_identical():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, 29623, q)) for r in range(2)]
    for p in procs:
        p.start()
    losses, spread = q.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert spread == 0.0 and losses[-1] < losses[0], (losses, spread)
